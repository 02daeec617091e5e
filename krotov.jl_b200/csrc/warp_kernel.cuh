// Persistent Krotov kernel for small Hilbert spaces, sm_100a: one warp per trajectory for d <= 32, two or four
// warps per trajectory (template parameter LPT = 64 / 128) for d <= 128 with narrow generator rows.
//
// One launch = one whole Krotov iteration (src/optimize.jl:279-371 of the reference):
//   backward sweep   chi_k(t_n) = exp(+i H_k^dagger dt) chi_k(t_{n+1})   stored for every n in HBM
//   forward sweep    per time step: overlaps Im<chi_k|mu_l|psi_k> -> grid-wide fixed-order sum
//                    -> pulse update -> Chebyshev step of every psi_k with the new pulse value
// with NO host round trip and NO kernel boundary between time steps.
//
// Mapping.  One group of LPT threads (a warp for d <= 32) owns one trajectory (or `tpw` of them), thread i owns
// component i of the state and row i of the generator.  The generator is kept as "G = 2c (H - beta)" rows in
// registers: W off-diagonal slots + the diagonal, rebuilt once per time step from the per-term
// rows P_t = 2c (H_t - beta delta_t0):  G = P_0 + sum_l eps_l[n] P_l.  The Chebyshev recursion
//   v_1 = G v_0 / 2,   v_j = G v_{j-1} + v_{j-2},   psi' = e^{-i beta dt} sum_j a_j v_j
// keeps v_{j-1}, v_{j-2} and the running sum in registers; only v_{j-1} is exchanged between
// lanes, through a 2-deep ping-pong buffer in shared memory (one __syncwarp per term).  Slots
// are assigned per matrix diagonal when the pattern allows it, so that every LDS.128 gather of
// a warp touches consecutive 16-byte words (bank-conflict free).
//
// Grid-wide reduction per time step (the serial dependency of Krotov's method): every CTA has a
// dedicated communication warp.  Trajectory warps leave their per-lane partial overlaps in
// shared memory and arrive on named barrier A; the comm warp reduces them in a fixed order,
// publishes the CTA partial into the step-indexed exchange array R[n][cta][l] (pre-filled with
// a NaN sentinel, so the 8-byte value is its own "ready" flag -- no fence, no atomics), polls
// the slots of all CTAs, sums them in a fixed order (bitwise reproducible),
// applies the update and releases the trajectory warps through named barrier B.  The gather is done
// by ONE reducer (the comm warp of CTA 0), which then broadcasts the L sums through E[n][l]; the other
// CTAs spin on that single line.  (An all-gather in which every CTA polled every slot made 147 CTAs
// hammer the same ~20 L2 lines and cost 7 us per step.)  That protocol is the fallback today: on one GPU the sum is
// an exact one-hop all-reduce through L2 integer atomics (atomic_grid_sum), and with several ranks every CTA adds its
// fixed-point partial into EVERY rank's accumulator over NVLink (xrank_atomic_sum) -- or, beyond a few hundred CTAs,
// the reducer pushes the rank's sum into every peer's mailbox (P2P stores) and the `world` mailbox slots are summed
// in rank order.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace kr {

constexpr int kMaxRanks = 8;
constexpr int kMaxCtrl = 8;
constexpr int kAmpMaxDeg = 4;
constexpr int kAmpRow = kAmpMaxDeg + 2;  // a row of WarpParams::amp_poly: kAmpMaxDeg+1 coefficients, then s_l
constexpr unsigned long long kSentinel = 0xFFFFFFFFFFFFFFFFull;

struct WarpParams {
    int d, N, L, N_T, n_gen;
    int wpc;   // trajectory warps per CTA (the CTA has wpc+1 warps)
    int tpw;   // trajectories per warp
    int nCTA;
    int mode;  // 0 = plain forward sweep under eps_old, 1 = full iteration
    int mu_hermitian;  // every control term of every generator is Hermitian (enables the idle-window precompute)
    int store_fw;
    int ndtc_f, ndtc_b, mmax_f, mmax_b;
    const int *gen_of_traj;
    const int *cols;           // [W][32] column (= smem index) of slot s for row `lane`
    const double2 *Pf, *Pb;    // [g][1+L][W+1][32], slot W = diagonal
    const double *inv_s_f;     // [g]  1/s_g = Delta_g/4 of the forward polynomial
    const double *coef_f, *coef_b;    // [g][ndtc][mmax]
    const int *m_f, *m_b;             // [g][ndtc]
    const double2 *phase_f, *phase_b; // [g][ndtc]  e^{-i beta dt}
    const int *dtc_f, *dtc_b;  // [N_T] dt class of every interval, per direction
    const double *dt;          // [N_T]
    const double *alpha;       // [L][N_T]  S_l[n] / lambda_l
    const double *eps_old;     // [L][N_T]
    double *eps_new;           // [L][N_T]
    // Non-linear control amplitudes (src/optimize.jl:268-272, 337-346): term l enters the generator with the coefficient
    // a_l(eps, n) = amp_shape[l][n] * sum_p amp_poly[l][p] eps^p.  The generator of a sweep under KNOWN pulses reads
    // amp_old = a(eps_old) (== eps_old for linear controls); mu_l = a_l'(eps_old) H_l scales the overlap sum by amp_dfac;
    // the forward step gets a(eps_new) from the comm warp.  All null / aliased for linear controls.
    const double *amp_old;     // [L][N_T]
    const double *amp_dfac;    // [L][N_T] or nullptr
    const double *amp_poly;    // [L][kAmpRow] (coefficients, then s_l: see amp_eval_cold) or nullptr
    const double *amp_shape;   // [L][N_T] or nullptr
    double *g_a_int;           // [L]
    double2 *X;                // [N][N_T+1][32]  chi trajectory, trajectory-major
    double2 *Phi;              // [N][N_T+1][32]  optional forward storage
    const double2 *psi0;       // [N][32]
    const double2 *target;     // [N][32]
    const double2 *chiT;       // [N][32] host-supplied boundary or nullptr
    const double2 *chi_coef;   // [N]
    double2 *psi_final;        // [N][32]
    double2 *tau;              // [N]
    double *R;                 // [N_T][L][nCTA] CTA partial sums, sentinel-filled before every iteration
    double *E;                 // [N_T][L] grid-wide sums broadcast by the reducer (CTA 0), sentinel-filled
    unsigned long long *acc;   // [N_T][L][3] fixed-point accumulators of the one-hop grid sum (zero-filled), or nullptr
    int mbox_all;              // several ranks: 1 = every CTA polls the rank's mailbox, 0 = the reducer polls it and broadcasts through E
    int rank, world;
    double *mbox[kMaxRanks];   // mailbox of every rank (this iteration's parity): [N_T][world][L]
    unsigned long long *xacc[kMaxRanks];  // several ranks, one-hop sum: fixed-point accumulators of EVERY rank (this
                               // iteration's parity, zero-filled): word (n, l, limb) at [((n*L + l)*4 + limb) * xacc_stride]
    int xacc_stride;           // distance between accumulator words in 8-byte units (1: one line per step, 16: one line per word)
    int xchg_hier;             // several ranks: 1 = hierarchical sum (rank sum in `acc`, then one add per rank into xacc)
    int total_ctas;            // CTAs of all ranks = arrivals per accumulator word
    int *err_flag;
    long long timeout_cycles;
    long long *prof;           // optional [nCTA][8] cycle counters (KROTOV_PROF=1), see krotov_get_profile
    // Tied control terms (krotov_set_control_terms): [L] control of every term (as doubles), then [L][N_T] a_t'(eps_old);
    // amp_dfac then holds ones, so that the comm warp's loop applies alpha_t to the control's du (see tie_sum_cold).
    // nullptr: every term is its own control.
    const double *tie;
    // several ranks emulated by ONE cooperative launch on one device (krotov_group_iterate: the multi-rank protocols
    // on a single-GPU box; ranks as separate launches on one GPU may never be co-resident): the launch parameter then
    // only carries `emul`, the per-rank parameter blocks in device memory, and CTA b serves the rank whose
    // [cta_base, cta_base + nCTA) holds b
    const WarpParams *emul;
    int emul_ranks, cta_base;
    // Replicated forward sweep (several ranks, every rank holds ALL trajectories): the backward sweep is sharded -- this
    // rank propagates trajectories [bw_lo, bw_hi) and writes every chi_k(t_n) into the chi trajectory of EVERY rank
    // (peer stores over NVLink) -- one rank barrier follows, and the time-serial forward sweep runs on every rank over all
    // trajectories with the one-rank exchange: no NVLink hop per time step, bit-identical replicas by construction.
    int rf_world, rf_rank, bw_lo, bw_hi;
    double2 *Xr[kMaxRanks];                 // chi trajectory of every rank (this iteration's parity); Xr[rf_rank] == X
    unsigned long long *rf_flag[kMaxRanks]; // [world] per rank: "rank r has finished its backward sweep of iteration i"
    unsigned int *rf_count;                 // arrivals of this rank's trajectory warps (zeroed per launch)
    unsigned long long rf_iter;
    // forwarder warps: the trajectory warps of a CTA that have no trajectory in the backward shard take the chi values of
    // the producing warps out of a shared-memory ring and store them to every rank, so the producers' serial chain carries
    // no peer store at all (0 = every producer stores to all ranks itself)
    int rf_fwd;
    int skip_bw;  // mode 1 in the REGULAR instances: the backward sweep was done by an RF instance (stage 1 of the replicated
                  // forward sweep); run the sequential update / forward sweep of the iteration only
    int rf_stride;  // RF instances: warp w plays slot (w * rf_stride) % wpc of the producer / forwarder roles (1 = identity)
    int rf_pack;  // producers per CTA when the backward shard is packed (warps of a CTA take CONSECUTIVE trajectories); 0 = spread
};

constexpr int kRfRing = 8;  // ring slots per producing warp (one chi record of 32 entries each)

__device__ __forceinline__ int ld_acquire_cta_shared(const int *a) {
    int v;
    asm volatile("ld.acquire.cta.shared.u32 %0, [%1];" : "=r"(v) : "r"((unsigned)__cvta_generic_to_shared(a)) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_cta_shared(int *a, const int v) {
    asm volatile("st.release.cta.shared.u32 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(a)), "r"(v) : "memory");
}
// shared-memory barrier objects: the "record ready" signal of the replicated forward sweep's rings.  A forwarder waiting in
// mbarrier.try_wait is suspended by the hardware; a polling loop with nanosleep was measured to come back every ~33 cycles
// (ncu: 38 M polls in one backward sweep, 30 % of the issue slots of the sub-partition it shares with a producing warp)
__device__ __forceinline__ void rf_mbar_init(unsigned long long *bar, const int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(count));
}
__device__ __forceinline__ void rf_mbar_arrive(unsigned long long *bar) {  // (release at CTA scope)
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"((unsigned)__cvta_generic_to_shared(bar)) : "memory");
}
__device__ __forceinline__ bool rf_mbar_try_wait(unsigned long long *bar, const unsigned parity) {  // (acquire at CTA scope)
    unsigned ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"((unsigned)__cvta_generic_to_shared(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}

template <bool EMUL>
__device__ __forceinline__ const WarpParams &select_params(const WarpParams &p0) {
    if (!EMUL) return p0;
    const WarpParams *q = p0.emul;
    for (int r = 0; r + 1 < p0.emul_ranks && (int)blockIdx.x >= q->cta_base + q->nCTA; ++r) ++q;
    return *q;
}

__device__ __forceinline__ void st_relaxed_f64(double *p, double v) {
    asm volatile("st.relaxed.sys.global.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_relaxed_u64(const double *p) {
    unsigned long long v;
    asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void bar_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ void bar_arrive(int id, int n) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(n) : "memory"); }

// acc += G_row . v   (complex).  Two independent FMA chains per component: with 4 chains in flight a
// warp already issues one DFMA every 2 cycles (the FP64 pipe rate measured on B200, tools/microbench.cu;
// dependent latency 8 cycles), so more chains only add the instructions that join them.
template <int W>
__device__ __forceinline__ void row_dot(const double2 (&g)[W + 1], const int (&col)[W], const double2 *__restrict__ vs,
                                        const double2 own, double &ar, double &ai) {
    double ar1 = 0.0, ai1 = 0.0;
    ar = fma(g[W].x, own.x, ar);
    ar1 = fma(-g[W].y, own.y, ar1);
    ai = fma(g[W].x, own.y, ai);
    ai1 = fma(g[W].y, own.x, ai1);
#pragma unroll
    for (int s = 0; s < W; ++s) {
        const double2 x = vs[col[s]];
        ar = fma(g[s].x, x.x, ar);
        ar1 = fma(-g[s].y, x.y, ar1);
        ai = fma(g[s].x, x.y, ai);
        ai1 = fma(g[s].y, x.x, ai1);
    }
    ar += ar1;
    ai += ai1;
}

// A trajectory is owned by a group of LPT threads (one generator row per thread): a warp for d <= 32, two or
// four warps for d <= 64 / 128.  Groups wider than a warp synchronise on their own named barrier.
template <int LPT>
__device__ __forceinline__ void grp_sync(const int bar_id) {
    if (LPT == 32)
        __syncwarp();
    else
        asm volatile("bar.sync %0, %1;" ::"r"(bar_id), "n"(LPT) : "memory");
}

template <int W, int LPT = 32>
__device__ __forceinline__ void load_row(const double2 *__restrict__ base, double2 (&out)[W + 1], int lane) {
#pragma unroll
    for (int s = 0; s <= W; ++s) out[s] = base[s * LPT + lane];
}

// One Chebyshev step.  v0buf holds psi for all lanes (written + synced by the caller).
template <int W, int LPT = 32>
__device__ __forceinline__ double2 cheby_step(const double2 psi, const double2 (&g)[W + 1], const int (&col)[W],
                                              const double2 *v0buf, double2 *bufA, double2 *bufB,
                                              const double *__restrict__ a, const int m, const double2 phase,
                                              const int lane, const int bar_id = 0) {
    double2 vm2 = psi;
    const double a0 = a[0];
    double outr = a0 * psi.x, outi = a0 * psi.y;
    double ar = 0.0, ai = 0.0;
    row_dot<W>(g, col, v0buf, psi, ar, ai);
    double2 vm1 = make_double2(0.5 * ar, 0.5 * ai);
    if (m > 1) {
        const double a1 = a[1];
        outr = fma(a1, vm1.x, outr);
        outi = fma(a1, vm1.y, outi);
    }
    bufB[lane] = vm1;
    grp_sync<LPT>(bar_id);
    double2 *cur = bufB, *nxt = bufA;
    for (int j = 2; j < m; ++j) {
        const double aj = a[j];
        ar = vm2.x;
        ai = vm2.y;
        row_dot<W>(g, col, cur, vm1, ar, ai);
        outr = fma(aj, ar, outr);
        outi = fma(aj, ai, outi);
        vm2 = vm1;
        vm1 = make_double2(ar, ai);
        nxt[lane] = vm1;
        grp_sync<LPT>(bar_id);
        double2 *t = cur;
        cur = nxt;
        nxt = t;
    }
    return make_double2(phase.x * outr - phase.y * outi, phase.x * outi + phase.y * outr);
}

// Per-step propagator metadata (coefficient count, final phase, coefficient row).  It is fetched ONE STEP
// AHEAD: the dependent chain dt-class -> (m, phase, row) is three L1/L2 round trips that would otherwise
// sit at the head of every time step.
struct StepMeta {
    int m;
    double2 phase;
    const double *a;
};
__device__ __forceinline__ StepMeta load_meta(const int *dtc, const int *m_tab, const double2 *ph_tab,
                                              const double *coef, int ndtc, int mmax, int gi, int n) {
    const int ci = gi * ndtc + dtc[n];
    StepMeta s;
    s.m = m_tab[ci];
    s.phase = ph_tab[ci];
    s.a = coef + (size_t)ci * mmax;
    return s;
}

// One truncated-Taylor step with scaling (Al-Mohy & Higham 2011; prop_method=Expmv): the rows g hold
// R = -i scale (H(eps) - mu) and a[j] = (dt / (scale s))^j / j!, so that each of the s repeats applies
//   v <- e^{-i mu dt/s} sum_{j<m} a_j R^j v  =  e^{-i mu dt/s} sum_{j<m} B^j / j! v,   B = -i dt/s (H - mu).
// m and s are fixed per (generator, dt class): (m-1) s products, no early termination, so the instruction stream and
// the bits are the same on every CTA and rank.  Same buffers as cheby_step: v0buf holds psi (written + synced by the
// caller); every product reads the buffer written behind the previous one and writes the other.
template <int W, int LPT = 32>
__device__ __forceinline__ double2 taylor_step(const double2 psi, const double2 (&g)[W + 1], const int (&col)[W],
                                               const double2 *v0buf, double2 *bufA, double2 *bufB,
                                               const double *__restrict__ a, const int m, const int s,
                                               const double2 phase, const int lane, const int bar_id = 0) {
    double2 v = psi;
    const double2 *cur = v0buf;
    double2 *nxt = bufB, *oth = bufA;
    for (int r = 0; r < s; ++r) {
        const double a0 = a[0];
        double outr = a0 * v.x, outi = a0 * v.y;
        double2 vj = v;
        for (int j = 1; j < m; ++j) {
            double ar = 0.0, ai = 0.0;
            row_dot<W>(g, col, cur, vj, ar, ai);
            const double aj = a[j];
            outr = fma(aj, ar, outr);
            outi = fma(aj, ai, outi);
            vj = make_double2(ar, ai);
            // behind the last product of a repeat the buffer takes the next repeat's input
            if (j + 1 == m) vj = make_double2(phase.x * outr - phase.y * outi, phase.x * outi + phase.y * outr);
            double2 *const w = nxt;
            w[lane] = vj;
            grp_sync<LPT>(bar_id);
            cur = w;
            nxt = oth;
            oth = w;
        }
        v = (m > 1) ? vj : make_double2(phase.x * outr - phase.y * outi, phase.x * outi + phase.y * outr);
    }
    return v;
}

// Taylor tables: m_tab holds (m, s) per (generator, dt class)
struct TaylorMeta {
    int m, s;
    double2 phase;
    const double *a;
};
__device__ __forceinline__ TaylorMeta load_meta_taylor(const int *dtc, const int *ms_tab, const double2 *ph_tab,
                                                       const double *coef, int ndtc, int mmax, int gi, int n) {
    const int ci = gi * ndtc + dtc[n];
    TaylorMeta s;
    const int2 ms = reinterpret_cast<const int2 *>(ms_tab)[ci];
    s.m = ms.x;
    s.s = ms.y;
    s.phase = ph_tab[ci];
    s.a = coef + (size_t)ci * mmax;
    return s;
}

// the step of the kernel's propagator: Chebyshev (StepMeta) or Taylor (TaylorMeta)
template <bool TAYLOR>
struct Prop {
    using Meta = StepMeta;
    static __device__ __forceinline__ Meta load(const int *dtc, const int *m_tab, const double2 *ph_tab, const double *coef,
                                                int ndtc, int mmax, int gi, int n) {
        return load_meta(dtc, m_tab, ph_tab, coef, ndtc, mmax, gi, n);
    }
    template <int W, int LPT>
    static __device__ __forceinline__ double2 step(const double2 psi, const double2 (&g)[W + 1], const int (&col)[W],
                                                   const double2 *v0buf, double2 *bufA, double2 *bufB, const Meta &mt,
                                                   const int lane, const int bar_id) {
        return cheby_step<W, LPT>(psi, g, col, v0buf, bufA, bufB, mt.a, mt.m, mt.phase, lane, bar_id);
    }
};
template <>
struct Prop<true> {
    using Meta = TaylorMeta;
    static __device__ __forceinline__ Meta load(const int *dtc, const int *m_tab, const double2 *ph_tab, const double *coef,
                                                int ndtc, int mmax, int gi, int n) {
        return load_meta_taylor(dtc, m_tab, ph_tab, coef, ndtc, mmax, gi, n);
    }
    template <int W, int LPT>
    static __device__ __forceinline__ double2 step(const double2 psi, const double2 (&g)[W + 1], const int (&col)[W],
                                                   const double2 *v0buf, double2 *bufA, double2 *bufB, const Meta &mt,
                                                   const int lane, const int bar_id) {
        return taylor_step<W, LPT>(psi, g, col, v0buf, bufA, bufB, mt.a, mt.m, mt.s, mt.phase, lane, bar_id);
    }
};

// Same recursion, but the first term v_1 = G v_0 / 2 was assembled by the caller from products that do not
// depend on the pulse value (computed while the warp waited for the grid-wide sum).
template <int W, int LPT = 32>
__device__ __forceinline__ double2 cheby_step_from_v1(const double2 psi, const double2 v1, const double2 (&g)[W + 1],
                                                      const int (&col)[W], double2 *bufA, double2 *bufB,
                                                      const double *__restrict__ a, const int m, const double2 phase,
                                                      const int lane, const int bar_id = 0) {
    double2 vm2 = psi, vm1 = v1;
    double outr = a[0] * psi.x, outi = a[0] * psi.y;
    if (m > 1) {
        const double a1 = a[1];
        outr = fma(a1, vm1.x, outr);
        outi = fma(a1, vm1.y, outi);
    }
    bufB[lane] = vm1;
    grp_sync<LPT>(bar_id);
    double2 *cur = bufB, *nxt = bufA;
    for (int j = 2; j < m; ++j) {
        const double aj = a[j];
        double ar = vm2.x, ai = vm2.y;
        row_dot<W>(g, col, cur, vm1, ar, ai);
        outr = fma(aj, ar, outr);
        outi = fma(aj, ai, outi);
        vm2 = vm1;
        vm1 = make_double2(ar, ai);
        nxt[lane] = vm1;
        grp_sync<LPT>(bar_id);
        double2 *t = cur;
        cur = nxt;
        nxt = t;
    }
    return make_double2(phase.x * outr - phase.y * outi, phase.x * outi + phase.y * outr);
}

__device__ __forceinline__ double warp_sum_xor(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ void st_relaxed_gpu_f64(double *p, double v) {
    asm volatile("st.relaxed.gpu.global.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory");
}
template <bool SYS>
__device__ __forceinline__ unsigned long long ld_poll_u64(const double *p) {
    unsigned long long v;
    if (SYS)
        asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    else
        asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

constexpr int kGatherMax = 40;  // ceil(kMaxCtrl * 148 / 32) = 37 values per lane at most

// Reducer side.  Gather `L*cnt` doubles laid out [l][c] at `base` (all loads of a round are in flight
// before any is examined; the round is repeated until no slot holds the sentinel), park them in shared
// memory and sum every control's `cnt` values in a FIXED order: the 32 lanes are split into groups of
// `G = 32 / pow2ceil(L)` lanes, group l sums control l -- lane j of the group adds c = j, j+G, j+2G, ...
// in order, then an xor butterfly inside the group.  Returns du[l] in tot[l] on every lane.
template <bool SYS>
__device__ __forceinline__ void reducer_gather(const double *base, const int cnt, const int L, const int lane,
                                               double *gbuf, double (&tot)[kMaxCtrl], int *err_flag,
                                               const long long timeout) {
    const int total = L * cnt;
    const int nper = (total + 31) >> 5;  // values per lane
    const long long t0 = clock64();
    int spins = 0;
    for (;;) {
        bool pending = false;
        for (int jb = 0; jb < nper; jb += 12) {  // 12 loads in flight per lane per batch (384 slots)
            unsigned long long u[12];
#pragma unroll
            for (int j = 0; j < 12; ++j) {
                const int idx = lane + 32 * (jb + j);
                u[j] = ld_poll_u64<SYS>(base + (idx < total ? idx : 0));
            }
#pragma unroll
            for (int j = 0; j < 12; ++j) {
                const int idx = lane + 32 * (jb + j);
                pending |= (u[j] == kSentinel);
                if (idx < total) gbuf[idx] = __longlong_as_double((long long)u[j]);
            }
        }
        if (!__any_sync(0xffffffffu, pending)) break;
        if ((++spins & 63) == 0) {
            if (clock64() - t0 > timeout || *(volatile int *)err_flag) {
                atomicExch(err_flag, 1);
                break;
            }
        }
    }
    __syncwarp();
    int p2 = 1;
    while (p2 < L) p2 <<= 1;
    const int G = 32 / p2;          // lanes per control
    const int myl = lane / G;       // control this lane works for
    const int j0 = lane - myl * G;
    double sacc = 0.0;
    if (myl < L)
        for (int c = j0; c < cnt; c += G) sacc += gbuf[myl * cnt + c];
    for (int o = G >> 1; o > 0; o >>= 1) sacc += __shfl_xor_sync(0xffffffffu, sacc, o);
#pragma unroll
    for (int l = 0; l < kMaxCtrl; ++l) tot[l] = __shfl_sync(0xffffffffu, sacc, (l < L ? l : 0) * G);
    __syncwarp();
}

// Everyone else: spin on the L broadcast words E[n][0..L-1] written by the reducer.  (Keeping several
// staggered poll loads in flight was measured and does not help: the wait is dominated by the two L2
// signalling hops, 690 cycles same-die / 1075 cross-die each, tools/pingpong.cu.)
__device__ __forceinline__ void poll_broadcast(const double *E, const int L, const int lane, double (&tot)[kMaxCtrl],
                                               int *err_flag, const long long timeout) {
    const long long t0 = clock64();
    int spins = 0;
    unsigned long long u;
    for (;;) {
        u = ld_poll_u64<false>(E + (lane < L ? lane : 0));
        if (__all_sync(0xffffffffu, u != kSentinel)) break;
        if ((++spins & 63) == 0) {
            if (clock64() - t0 > timeout || *(volatile int *)err_flag) {
                atomicExch(err_flag, 1);
                break;
            }
        }
    }
    const double v = __longlong_as_double((long long)u);
#pragma unroll
    for (int l = 0; l < kMaxCtrl; ++l) tot[l] = __shfl_sync(0xffffffffu, v, l < L ? l : 0);
}


// ---- exact one-hop grid sum through L2 integer atomics ---------------------------------------------------------
// Every CTA converts its partial sum to a 120-bit fixed-point number (unit 2^-88, bias 2^119), splits it into three
// 40-bit limbs and adds limb j into word j of the step's accumulator with ONE red.add.u64 each; the same add bumps an
// arrival count in the word's top byte (and a "does not fit" count in the byte below).  Integer addition is
// associative, so the total is the EXACT sum of the CTA partials whatever the arrival order -- bitwise reproducible
// like the fixed-order gather, but in one L2 hop instead of two (CTA -> reducer -> everybody): every CTA polls the
// L*3 words (one 64-byte line for two controls) until each carries all arrivals, then rounds the sum to double once.
// tools/atomic_allreduce.cu: 1529 cycles per round at 148 CTAs against 2356 for gather + broadcast.
// A partial that is not finite or not below 2^31 marks the step and all CTAs redo it with the gather protocol.
constexpr int kFixFrac = 88, kFixLimbBits = 40, kFixLimbs = 3, kFixBiasBit = 119;

__device__ __forceinline__ bool fix_from_double(const double x, unsigned __int128 &biased, const int lim_exp = 31) {
    const unsigned long long bits = (unsigned long long)__double_as_longlong(fabs(x));
    const int ebits = (int)(bits >> 52);
    if (ebits >= 1023 + lim_exp) return false;  // |x| >= 2^lim_exp, Inf or NaN
    const unsigned long long mant = (bits & 0xFFFFFFFFFFFFFull) | (ebits ? (1ull << 52) : 0ull);
    const int shift = (ebits ? ebits : 1) - 1075 + kFixFrac;  // |x| = mant * 2^(shift - kFixFrac)
    unsigned __int128 mag = 0;
    if (shift >= 0)
        mag = (unsigned __int128)mant << shift;
    else if (shift > -64)
        mag = mant >> (-shift);  // below 2^-88: truncated
    const unsigned __int128 bias = (unsigned __int128)1 << kFixBiasBit;
    biased = (x < 0.0) ? bias - mag : bias + mag;
    return true;
}

// sum of `n` biased numbers (limb sums w0, w1, w2 without their count bytes) -> double, rounded to nearest once
__device__ __forceinline__ double fix_to_double(const unsigned long long w0, const unsigned long long w1,
                                                const unsigned long long w2, const int n) {
    const unsigned long long mask = (1ull << 48) - 1;
    unsigned __int128 sum = (unsigned __int128)(w0 & mask) + ((unsigned __int128)(w1 & mask) << kFixLimbBits) +
                            ((unsigned __int128)(w2 & mask) << (2 * kFixLimbBits));
    const unsigned __int128 bias = (unsigned __int128)n << kFixBiasBit;
    const bool neg = sum < bias;
    const unsigned __int128 mag = neg ? bias - sum : sum - bias;
    const unsigned long long hi = (unsigned long long)(mag >> 64), lo = (unsigned long long)mag;
    double d;
    if (hi == 0) {
        d = __ull2double_rn(lo);
    } else {
        const int sh = 64 - __clzll((long long)hi);  // 1..64 bits live in `hi`
        unsigned long long top = (sh == 64) ? hi : ((hi << (64 - sh)) | (lo >> sh));
        const unsigned long long lost = (sh == 64) ? lo : (lo << (64 - sh));
        if (lost) top |= 1ull;  // sticky bit, 11 places below the rounding position
        d = scalbn(__ull2double_rn(top), sh);
    }
    d = scalbn(d, -kFixFrac);
    return neg ? -d : d;
}

__device__ __forceinline__ void red_add_u64(unsigned long long *p, unsigned long long v) {
    asm volatile("red.relaxed.gpu.global.add.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// Returns true when tot[] holds the grid-wide sums; false when some CTA's partial did not fit (all CTAs see the same
// verdict) and the step has to be redone with the gather protocol.
__device__ __forceinline__ bool atomic_grid_sum(unsigned long long *An, const int nCTA, const int L, const int lane,
                                                double (&tot)[kMaxCtrl], int *err_flag, const long long timeout,
                                                const bool wait = true) {
    const int nw = L * kFixLimbs;           // words of this step; lane q < nw owns word q = (control q / 3, limb q % 3)
    const int myl = lane / kFixLimbs, myj = lane - myl * kFixLimbs;
    double mine = 0.0;
#pragma unroll
    for (int l = 0; l < kMaxCtrl; ++l)
        if (l == myl) mine = tot[l];
    if (lane < nw) {
        unsigned __int128 v;
        const bool ok = fix_from_double(mine, v);
        unsigned long long add = 1ull << 56;  // one arrival
        if (ok)
            add += (unsigned long long)(v >> (myj * kFixLimbBits)) & ((1ull << kFixLimbBits) - 1);
        else
            add += 1ull << 48;  // one partial that does not fit
        red_add_u64(An + lane, add);
    }
    if (!wait) return true;  // contributor only (several ranks: the reducer alone needs the rank's sum)
    const long long t0 = clock64();
    int spins = 0;
    unsigned long long w = 0;
    for (;;) {
        if (lane < nw) w = ld_poll_u64<false>(reinterpret_cast<const double *>(An + lane));
        const bool pending = lane < nw && (int)(w >> 56) != nCTA;
        if (!__any_sync(0xffffffffu, pending)) break;
        if ((++spins & 63) == 0) {
            if (clock64() - t0 > timeout || *(volatile int *)err_flag) {
                atomicExch(err_flag, 1);
                break;
            }
        }
    }
    const bool misfit = lane < nw && ((w >> 48) & 0xFF) != 0;
    if (__any_sync(0xffffffffu, misfit)) return false;
    // lane l < L rebuilds control l from its three words
    const int src = (lane < L ? lane : 0) * kFixLimbs;
    const unsigned long long w0 = __shfl_sync(0xffffffffu, w, src), w1 = __shfl_sync(0xffffffffu, w, src + 1),
                             w2 = __shfl_sync(0xffffffffu, w, src + 2);
    const double du = fix_to_double(w0, w1, w2, nCTA);
#pragma unroll
    for (int l = 0; l < kMaxCtrl; ++l) tot[l] = __shfl_sync(0xffffffffu, du, l < L ? l : 0);
    return true;
}

// ---- the same sum across SEVERAL ranks in one NVLink hop ---------------------------------------------------------
// Every CTA of every rank adds its fixed-point partial into the step's accumulator of EVERY rank (local L2 atomics and
// `red.add.u64` over NVLink into the peers' memory, fire and forget) and polls only its own rank's copy until it carries
// the arrivals of all CTAs of all ranks.  All copies receive the same set of integer adds, so every rank rounds the
// same exact sum: bit-identical pulses on all replicas without a reducer, a rank-ordered sum or a broadcast hop
// (CTA -> local reducer -> peers' mailboxes -> everybody becomes CTA -> everybody).  Up to 2047 arrivals: the number
// is 117 bits wide (unit 2^-88, bias 2^116, |partial| < 2^28) in four 30-bit limbs; word = limb sum (41 bits) |
// "does not fit" count (11 bits) | arrival count (12 bits).  A misfit makes every CTA of every rank redo the step
// with the mailbox protocol below (same verdict everywhere, because it is read from the same sums).
constexpr int kXLimbBits = 30, kXLimbs = 4, kXBiasBit = 116, kXMisShift = 41, kXCntShift = 52, kXMaxArrivals = 2047;

__device__ __forceinline__ bool fixx_from_double(const double x, unsigned __int128 &biased) {
    const unsigned long long bits = (unsigned long long)__double_as_longlong(fabs(x));
    const int ebits = (int)(bits >> 52);
    if (ebits >= 1023 + (kXBiasBit - kFixFrac)) return false;  // |x| >= 2^28, Inf or NaN
    const unsigned long long mant = (bits & 0xFFFFFFFFFFFFFull) | (ebits ? (1ull << 52) : 0ull);
    const int shift = (ebits ? ebits : 1) - 1075 + kFixFrac;
    unsigned __int128 mag = 0;
    if (shift >= 0)
        mag = (unsigned __int128)mant << shift;
    else if (shift > -64)
        mag = mant >> (-shift);
    const unsigned __int128 bias = (unsigned __int128)1 << kXBiasBit;
    biased = (x < 0.0) ? bias - mag : bias + mag;
    return true;
}

__device__ __forceinline__ double fix_mag_to_double(const unsigned __int128 mag, const bool neg) {
    const unsigned long long hi = (unsigned long long)(mag >> 64), lo = (unsigned long long)mag;
    double d;
    if (hi == 0) {
        d = __ull2double_rn(lo);
    } else {
        const int sh = 64 - __clzll((long long)hi);
        unsigned long long top = (sh == 64) ? hi : ((hi << (64 - sh)) | (lo >> sh));
        const unsigned long long lost = (sh == 64) ? lo : (lo << (64 - sh));
        if (lost) top |= 1ull;
        d = scalbn(__ull2double_rn(top), sh);
    }
    d = scalbn(d, -kFixFrac);
    return neg ? -d : d;
}

__device__ __forceinline__ void red_add_sys_u64(unsigned long long *p, unsigned long long v) {
    asm volatile("red.relaxed.sys.global.add.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

__device__ __forceinline__ bool xrank_atomic_sum(const WarpParams &p, const int n, const int L, const int lane,
                                                 double (&tot)[kMaxCtrl]) {
    const int nw = L * kXLimbs;  // <= 32: lane q owns word q = (control q / 4, limb q % 4)
    const int myl = lane / kXLimbs, myj = lane - myl * kXLimbs;
    double mine = 0.0;
#pragma unroll
    for (int l = 0; l < kMaxCtrl; ++l)
        if (l == myl) mine = tot[l];
    const size_t off = ((size_t)n * nw + (lane < nw ? lane : 0)) * (size_t)p.xacc_stride;
    if (lane < nw) {
        unsigned __int128 v;
        const bool ok = fixx_from_double(mine, v);
        unsigned long long add = 1ull << kXCntShift;
        if (ok)
            add += (unsigned long long)(v >> (myj * kXLimbBits)) & ((1ull << kXLimbBits) - 1);
        else
            add += 1ull << kXMisShift;
        for (int i = 1; i <= p.world; ++i) {  // peers first (the long way), own copy last
            int r = p.rank + i;
            if (r >= p.world) r -= p.world;
            red_add_sys_u64(p.xacc[r] + off, add);
        }
    }
    const long long t0 = clock64();
    int spins = 0;
    unsigned long long w = 0;
    const double *mine_p = reinterpret_cast<const double *>(p.xacc[p.rank] + off);
    for (;;) {
        if (lane < nw) w = ld_poll_u64<true>(mine_p);
        const bool pending = lane < nw && (int)(w >> kXCntShift) != p.total_ctas;
        if (!__any_sync(0xffffffffu, pending)) break;
        if ((++spins & 63) == 0) {
            if (clock64() - t0 > p.timeout_cycles || *(volatile int *)p.err_flag) {
                atomicExch(p.err_flag, 1);
                break;
            }
        }
    }
    const bool misfit = lane < nw && ((w >> kXMisShift) & 0x7FF) != 0;
    if (__any_sync(0xffffffffu, misfit)) return false;
    const int src = (lane < L ? lane : 0) * kXLimbs;
    const unsigned long long mask = (1ull << kXMisShift) - 1;
    unsigned __int128 sum = 0;
#pragma unroll
    for (int j = 0; j < kXLimbs; ++j)
        sum += (unsigned __int128)(__shfl_sync(0xffffffffu, w, src + j) & mask) << (j * kXLimbBits);
    const unsigned __int128 bias = (unsigned __int128)p.total_ctas << kXBiasBit;
    const bool neg = sum < bias;
    const double du = fix_mag_to_double(neg ? bias - sum : sum - bias, neg);
#pragma unroll
    for (int l = 0; l < kMaxCtrl; ++l) tot[l] = __shfl_sync(0xffffffffu, du, l < L ? l : 0);
    return true;
}

// ---- the sum across several ranks, hierarchical: local L2 atomics, then ONE add per rank and word over NVLink --------
// xrank_atomic_sum above makes every CTA of every rank add into every rank's accumulator: `total_ctas` atomics per word
// and time step land on one line of every rank (2048 for 8 x 32 CTAs and two controls), and the cost grows with the
// number of ranks.  Here every CTA adds its fixed-point partial (the 120-bit format of atomic_grid_sum, |partial| < 2^28)
// into its OWN rank's accumulator with `atom.add`, which returns the previous value: the lane whose add completes the
// arrival count of a word holds that word's exact rank sum and forwards it -- limb sum, one arrival, a misfit mark --
// into the same word of every rank's cross-rank accumulator with one `red.add.u64` each (peers over NVLink, fire and
// forget).  No CTA waits for the rank sum (the mailbox protocol's reducer does), there is no polling reducer, every rank
// receives `world` adds per word and step, and all ranks round the same exact integer sum: bit-identical pulses.
// Cross-rank word: limb sum (52 bits: 40 + 8 for <= 255 CTAs per rank + 4 for <= 8 ranks... here <= 2047 CTAs in total)
// | ranks with a misfit (4 bits) | rank arrivals (4 bits).
constexpr int kHSumBits = 52, kHMisShift = 52, kHCntShift = 56, kHLimExp = 28;

__device__ __forceinline__ unsigned long long atom_add_u64(unsigned long long *p, unsigned long long v) {
    unsigned long long old;
    asm volatile("atom.relaxed.gpu.global.add.u64 %0, [%1], %2;" : "=l"(old) : "l"(p), "l"(v) : "memory");
    return old;
}

__device__ __forceinline__ bool xrank_hier_sum(const WarpParams &p, const int n, const int L, const int lane,
                                               double (&tot)[kMaxCtrl]) {
    const int nw = L * kFixLimbs;  // lane q < nw owns word q = (control q / 3, limb q % 3)
    const int myl = lane / kFixLimbs, myj = lane - myl * kFixLimbs;
    double mine = 0.0;
#pragma unroll
    for (int l = 0; l < kMaxCtrl; ++l)
        if (l == myl) mine = tot[l];
    // cross-rank words live in the xacc area with its layout [(n * L + l) * 4 + limb] (the fourth limb slot is unused).
    // Store variant (xchg_hier == 2): every word has one 8-byte slot PER RANK, [((n * L + l) * 4 + limb) * 8 + rank], the
    // completing lane writes its rank's slot of every rank with a plain store (no NVLink atomic) and the pollers add the
    // `world` slots of a word themselves.
    const bool by_store = p.xchg_hier == 2;
    const size_t widx = ((size_t)n * L + (lane < nw ? myl : 0)) * kXLimbs + (lane < nw ? myj : 0);
    const size_t off = by_store ? widx * kMaxRanks : widx * (size_t)p.xacc_stride;
    if (lane < nw) {
        unsigned __int128 v;
        const bool ok = fix_from_double(mine, v, kHLimExp);
        unsigned long long add = 1ull << 56;  // one CTA arrival
        if (ok)
            add += (unsigned long long)(v >> (myj * kFixLimbBits)) & ((1ull << kFixLimbBits) - 1);
        else
            add += 1ull << 48;  // one partial that does not fit
        unsigned long long total = add;
        if (p.nCTA > 1) total += atom_add_u64(p.acc + (size_t)n * nw + lane, add);
        if ((int)(total >> 56) == p.nCTA) {  // this add completed the rank's word: forward the rank sum
            unsigned long long fwd = 1ull << kHCntShift;
            if ((total >> 48) & 0xFF)
                fwd += 1ull << kHMisShift;
            else
                fwd += total & ((1ull << 48) - 1);
            for (int i = 1; i <= p.world; ++i) {  // peers first (the long way), own copy last
                int r = p.rank + i;
                if (r >= p.world) r -= p.world;
                if (by_store)
                    asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p.xacc[r] + off + p.rank), "l"(fwd) : "memory");
                else
                    red_add_sys_u64(p.xacc[r] + off, fwd);
            }
        }
    }
    const long long t0 = clock64();
    int spins = 0;
    unsigned long long w = 0;
    const double *mine_p = reinterpret_cast<const double *>(p.xacc[p.rank] + off);
    for (;;) {
        bool pending = false;
        if (lane < nw) {
            if (by_store) {
                unsigned long long u[kMaxRanks];
#pragma unroll
                for (int r = 0; r < kMaxRanks; ++r) u[r] = (r < p.world) ? ld_poll_u64<true>(mine_p + r) : 0ull;
                w = 0;
#pragma unroll
                for (int r = 0; r < kMaxRanks; ++r) {
                    pending |= (r < p.world) && u[r] == 0ull;
                    w += u[r];
                }
            } else {
                w = ld_poll_u64<true>(mine_p);
                pending = (int)(w >> kHCntShift) != p.world;
            }
        }
        if (!__any_sync(0xffffffffu, pending)) break;
        if ((++spins & 63) == 0) {
            if (clock64() - t0 > p.timeout_cycles || *(volatile int *)p.err_flag) {
                atomicExch(p.err_flag, 1);
                break;
            }
        }
    }
    const bool misfit = lane < nw && ((w >> kHMisShift) & 0xF) != 0;
    if (__any_sync(0xffffffffu, misfit)) return false;
    // lane l < L rebuilds control l: the bias (2^119 per CTA = 2^39 in limb 2) comes off in the top limb, so the
    // magnitude (< total_ctas * 2^28 * 2^88) fits the signed 128-bit sum whatever the number of CTAs
    const int src = (lane < L ? lane : 0) * kFixLimbs;
    const unsigned long long mask = (1ull << kHSumBits) - 1;
    const unsigned long long w0 = __shfl_sync(0xffffffffu, w, src) & mask, w1 = __shfl_sync(0xffffffffu, w, src + 1) & mask,
                             w2 = __shfl_sync(0xffffffffu, w, src + 2) & mask;
    const long long top = (long long)w2 - ((long long)p.total_ctas << (kFixBiasBit - 2 * kFixLimbBits));
    const __int128 sum = ((__int128)top << (2 * kFixLimbBits)) + ((__int128)w1 << kFixLimbBits) + (__int128)w0;
    const bool neg = sum < 0;
    const double du = fix_mag_to_double((unsigned __int128)(neg ? -sum : sum), neg);
#pragma unroll
    for (int l = 0; l < kMaxCtrl; ++l) tot[l] = __shfl_sync(0xffffffffu, du, l < L ? l : 0);
    return true;
}

// ---- exchange paths that are kept OUT OF LINE ------------------------------------------------------------------------
// The comm warp's per-step loop used to carry every protocol inline: ~58 KB of code of which a step on one rank runs a
// few hundred bytes, spread between jumps over the rest.  That cost the single-CTA case a full microsecond per time
// step (instruction fetch; C3: 7.8 -> 10.1 ms per iteration as the protocols accumulated), so everything but the
// one-rank atomic sum now lives in two functions that are called, not inlined.  `tot` travels through local memory.

// Several ranks: hierarchical sum or one-hop sum, with the mailbox protocol as their fallback (and as a protocol of its
// own).  On return tot[] holds the sums over all CTAs of all ranks, the same bits on every CTA of every rank.
static __device__ __noinline__ void exchange_ranks(const WarpParams *pp, const int cta, const int n, const int L, const int lane,
                                            double *tot_io, double *gbuf) {
    const WarpParams &p = *pp;
    double tot[kMaxCtrl];
#pragma unroll
    for (int l = 0; l < kMaxCtrl; ++l) tot[l] = tot_io[l];
    bool summed = false, acc_used = false;
    if (p.xacc[0] != nullptr) {
        if (p.xchg_hier) {
            summed = xrank_hier_sum(p, n, L, lane, tot);
            acc_used = true;  // the rank's accumulator words of this step are spent
        } else {
            summed = xrank_atomic_sum(p, n, L, lane, tot);
        }
        if (!summed && cta == 0 && lane == 0) atomicAdd(p.err_flag + 1, 1);  // krotov_info.fallback_steps
    }
    if (!summed) {
        // ---- mailboxes.  Every CTA adds its partial into the rank's fixed-point accumulator (and leaves it in
        // R for the fallback); the reducer (CTA 0) alone waits for the exact rank sum, pushes it into the mailbox
        // of EVERY rank over NVLink, and every CTA of every rank polls its own rank's mailbox and adds the
        // `world` rank sums in rank order: identical bits everywhere, no broadcast hop behind the NVLink hop.
        double *Rn = p.R + (size_t)n * L * p.nCTA;
        const bool use_acc = p.acc != nullptr && p.nCTA > 1 && !acc_used;
        if (p.nCTA > 1) {
#pragma unroll
            for (int l = 0; l < kMaxCtrl; ++l)
                if (l < L && lane == l) st_relaxed_gpu_f64(Rn + (size_t)l * p.nCTA + cta, tot[l]);
        }
        bool have_rank_sum = p.nCTA == 1;
        if (use_acc)
            have_rank_sum = atomic_grid_sum(p.acc + (size_t)n * L * kFixLimbs, p.nCTA, L, lane, tot, p.err_flag,
                                            p.timeout_cycles, cta == 0);
        const size_t off = (size_t)n * L * p.world;  // mailbox layout [n][l][rank]
        if (cta == 0) {
            if (!have_rank_sum) {
                if (use_acc && lane == 0) atomicAdd(p.err_flag + 1, 1);  // krotov_info.fallback_steps
                reducer_gather<false>(Rn, p.nCTA, L, lane, gbuf, tot, p.err_flag, p.timeout_cycles);
            }
#pragma unroll
            for (int l = 0; l < kMaxCtrl; ++l)
                if (l < L && lane < p.world) st_relaxed_f64(p.mbox[lane] + off + (size_t)l * p.world + p.rank, tot[l]);
        }
        if (p.mbox_all || p.nCTA == 1) {
            reducer_gather<true>(p.mbox[p.rank] + off, p.world, L, lane, gbuf, tot, p.err_flag, p.timeout_cycles);
        } else {
            double *En = p.E + (size_t)n * L;
            if (cta == 0) {
                reducer_gather<true>(p.mbox[p.rank] + off, p.world, L, lane, gbuf, tot, p.err_flag, p.timeout_cycles);
#pragma unroll
                for (int l = 0; l < kMaxCtrl; ++l)
                    if (l < L && lane == l) st_relaxed_gpu_f64(En + l, tot[l]);
            } else {
                poll_broadcast(En, L, lane, tot, p.err_flag, p.timeout_cycles);
            }
        }
    }
#pragma unroll
    for (int l = 0; l < kMaxCtrl; ++l) tot_io[l] = tot[l];
}

// One rank, gather + broadcast: the protocol before the atomic sum existed, and its fallback when a partial does not
// fit the fixed-point range.  R[n][l][cta]: CTA partials; E[n][l]: the grid-wide sums, written by the reducer (CTA 0).
static __device__ __noinline__ void exchange_gather(const WarpParams *pp, const int cta, const int n, const int L, const int lane,
                                             double *tot_io, double *gbuf) {
    const WarpParams &p = *pp;
    double tot[kMaxCtrl];
#pragma unroll
    for (int l = 0; l < kMaxCtrl; ++l) tot[l] = tot_io[l];
    double *Rn = p.R + (size_t)n * L * p.nCTA;
    double *En = p.E + (size_t)n * L;
    if (cta != 0) {
#pragma unroll
        for (int l = 0; l < kMaxCtrl; ++l)
            if (l < L && lane == l) st_relaxed_gpu_f64(Rn + (size_t)l * p.nCTA + cta, tot[l]);
        poll_broadcast(En, L, lane, tot, p.err_flag, p.timeout_cycles);
    } else {
#pragma unroll
        for (int l = 0; l < kMaxCtrl; ++l)
            if (l < L && lane == l) st_relaxed_gpu_f64(Rn + (size_t)l * p.nCTA, tot[l]);
        reducer_gather<false>(Rn, p.nCTA, L, lane, gbuf, tot, p.err_flag, p.timeout_cycles);
#pragma unroll
        for (int l = 0; l < kMaxCtrl; ++l)
            if (l < L && lane == l) st_relaxed_gpu_f64(En + l, tot[l]);
    }
#pragma unroll
    for (int l = 0; l < kMaxCtrl; ++l) tot_io[l] = tot[l];
}

// a_l(e, n) = shape * sum_p poly[l][p] x^p, x = tanh(s_l e) where s_l > 0 (saturating amplitudes), else x = e
// (non-linear amplitudes only; kept out of the comm warp's loop body).  s_l travels in the polynomial's row rather than
// in a parameter field of its own: the function reads the same two fields as without saturation, and the comm warp's
// loop around its call site compiles to the same code.
static __device__ __noinline__ double amp_eval_cold(const WarpParams *pp, const int l, const double e, const double shp) {
    double c = e;
    if (pp->amp_poly != nullptr) {
        const double *q = pp->amp_poly + l * kAmpRow;
        const double x = q[kAmpMaxDeg + 1] != 0.0 ? tanh(q[kAmpMaxDeg + 1] * e) : e;
        c = q[kAmpMaxDeg];
#pragma unroll
        for (int d = kAmpMaxDeg - 1; d >= 0; --d) c = fma(c, x, q[d]);
    }
    if (pp->amp_shape != nullptr) c = __dmul_rn(shp, c);
    return c;
}

// Tied control terms: every lane of the comm warp passes the grid-wide overlap sum `s` of its term (lanes < L) and gets
// back du of the term's control, the sum over the control's terms in ascending t of a_t'(eps_old) s_t (the same bits on
// every lane of every CTA and rank: the inputs are).  Out of line, as amp_eval_cold.
static __device__ __noinline__ double tie_sum_cold(const WarpParams *pp, const int lane, const int n, const int L, const double s) {
    const double *ctrl = pp->tie, *dfac = pp->tie + L;
    const double v = lane < L ? __dmul_rn(dfac[(size_t)lane * pp->N_T + n], s) : 0.0;
    const double c = lane < L ? ctrl[lane] : -1.0;
    double du = 0.0;
    bool first = true;
#pragma unroll
    for (int t = 0; t < kMaxCtrl; ++t) {
        const double vt = __shfl_sync(0xffffffffu, v, t);
        if (t < L && ctrl[t] == c) {
            du = first ? vt : __dadd_rn(du, vt);
            first = false;
        }
    }
    return du;
}

// The communication warp of a CTA (shared by both kernel variants): per time step it waits for the CTA's
// per-lane partial overlaps (named barrier 1), reduces them in a fixed order, runs the grid / rank exchange,
// applies the pulse update (src/optimize.jl:351-358) and releases the trajectory warps (named barrier 2).
__device__ __forceinline__ void comm_warp_run(const WarpParams &p, const int cta, const int L, const int lane, const int wpc,
                                              const int nthr_all, double *red, double *eps_s, double *gbuf,
                                              WarpParams *p_sh) {
    const int N_T = p.N_T;
    if (p.mode != 1) return;
    // The out-of-line exchange functions read the parameter block through a pointer.  A pointer to the kernel
    // parameter itself is a generic address into the constant bank: every field read is a slow, uncached-path load
    // (measured: +0.35 us per time step on 2 GPUs).  They get a copy in shared memory instead.
    {
        const unsigned long long *src = reinterpret_cast<const unsigned long long *>(&p);
        unsigned long long *dst = reinterpret_cast<unsigned long long *>(p_sh);
        for (int i = lane; i < (int)(sizeof(WarpParams) / 8); i += 32) dst[i] = src[i];
        __syncwarp();
    }
    double ga = 0.0;  // lane l accumulates g_a_int[l]  (CTA 0 writes it)
    const bool nonlin = p.amp_dfac != nullptr;  // non-linear control amplitudes (rare): handled out of line
    const bool tied = p.tie != nullptr;         // tied control terms (rare, implies nonlin): handled out of line
    long long c_wait_a = 0, c_reduce = 0, c_gather = 0;
    for (int n = 0; n < N_T; ++n) {
        double a_ln = 0.0, e_old = 0.0, dtn = 0.0, dfac = 1.0, shp = 1.0, a_eff = 0.0;
        if (lane < L) {
            a_ln = p.alpha[(size_t)lane * N_T + n];
            e_old = p.eps_old[(size_t)lane * N_T + n];
            dtn = p.dt[n];
            a_eff = a_ln;
            if (nonlin) {  // fetched and folded BEFORE the barrier: nothing of it sits behind the exchange
                dfac = p.amp_dfac[(size_t)lane * N_T + n];
                if (p.amp_shape != nullptr) shp = p.amp_shape[(size_t)lane * N_T + n];
                a_eff = __dmul_rn(a_ln, dfac);
            }
        }
        const long long c0 = clock64();
        bar_sync(1, nthr_all);  // barrier A: partials are in `red`
        const long long c1 = clock64();
        double tot[kMaxCtrl];
#pragma unroll
        for (int l = 0; l < kMaxCtrl; ++l) {
            double sacc = 0.0;
            if (l < L)
                for (int q = 0; q < wpc; ++q) sacc += red[(size_t)l * wpc * 32 + q * 32 + lane];
            tot[l] = sacc;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
            for (int l = 0; l < kMaxCtrl; ++l)
                if (l < L) tot[l] += __shfl_xor_sync(0xffffffffu, tot[l], o);
        }
        const long long c2 = clock64();
        bool summed = p.nCTA == 1 && p.world == 1;
        if (p.world > 1) {
            double tl[kMaxCtrl];
#pragma unroll
            for (int l = 0; l < kMaxCtrl; ++l) tl[l] = tot[l];
            exchange_ranks(p_sh, cta, n, L, lane, tl, gbuf);
#pragma unroll
            for (int l = 0; l < kMaxCtrl; ++l) tot[l] = tl[l];
            summed = true;
        } else if (p.acc != nullptr && p.nCTA > 1) {
            summed = atomic_grid_sum(p.acc + (size_t)n * L * kFixLimbs, p.nCTA, L, lane, tot, p.err_flag, p.timeout_cycles);
            if (!summed && cta == 0 && lane == 0) atomicAdd(p.err_flag + 1, 1);  // krotov_info.fallback_steps
        }
        if (!summed) {
            double tl[kMaxCtrl];
#pragma unroll
            for (int l = 0; l < kMaxCtrl; ++l) tl[l] = tot[l];
            exchange_gather(p_sh, cta, n, L, lane, tl, gbuf);
#pragma unroll
            for (int l = 0; l < kMaxCtrl; ++l) tot[l] = tl[l];
        }
        const long long c3 = clock64();
        c_wait_a += c1 - c0;
        c_reduce += c2 - c1;
        c_gather += c3 - c2;
        double mine = 0.0;  // lane l holds du[l]
#pragma unroll
        for (int l = 0; l < kMaxCtrl; ++l)
            if (lane == l) mine = tot[l];
        if (tied) mine = tie_sum_cold(p_sh, lane, n, L, mine);  // (amp_dfac holds ones: a_eff = alpha, du = mine)
        double e_new = 0.0;
        if (lane < L) {
            const double d_eps = __dmul_rn(a_eff, mine);     // src/optimize.jl:355 (a_eff = alpha, or alpha a_l' when non-linear)
            e_new = __dadd_rn(e_old, d_eps);                 // :356
            double c_new = e_new;                            // coefficient of H_l in the forward step
            if (nonlin) c_new = amp_eval_cold(p_sh, lane, e_new, shp);
            eps_s[lane] = c_new;
        }
        bar_arrive(2, nthr_all);  // barrier B: eps_s is valid
        if (cta == 0 && lane < L) {  // bookkeeping, off the critical path
            p.eps_new[(size_t)lane * N_T + n] = e_new;
            const double du = nonlin ? __dmul_rn(dfac, mine) : mine;  // mu_l = a_l'(eps^(i)_l[n]) H_l  (:337-346)
            ga = __dadd_rn(ga, __dmul_rn(__dmul_rn(a_ln, __dmul_rn(fabs(du), fabs(du))), dtn));  // :357
        }
    }
    if (cta == 0 && lane < L) p.g_a_int[lane] = ga;
    if (p.prof != nullptr && lane == 0) {
        p.prof[cta * 8 + 3] = c_wait_a;
        p.prof[cta * 8 + 4] = c_reduce;
        p.prof[cta * 8 + 5] = c_gather;
    }
}

// ---- replicated forward sweep: the cold parts, out of line so that the sweeps of the RF instances keep the code of the
// regular ones (the parameter block is read through a generic pointer here: slow loads, off every critical path)
// Forwarder warp: takes the chi records of its producing warps out of their rings and stores them to every rank.
static __device__ __noinline__ void rf_forward_records(const WarpParams *pp, const double2 *rf_ring, unsigned long long *rf_bar,
                                                       int *rf_prog, const int cta, const int warp, const int lane,
                                                       const int n_prod, const int n_fwd) {
    const WarpParams &p = *pp;
    const int N_T = p.N_T, wpc = p.wpc, world = p.rf_world, nCTA = p.nCTA, bw_lo = p.bw_lo;
    const long long timeout = p.timeout_cycles;
    double2 *Xr[kMaxRanks];
#pragma unroll
    for (int r = 0; r < kMaxRanks; ++r) Xr[r] = p.Xr[r];
    const long long t0 = clock64();
    bool dead = false;
    for (int i = 0; i <= N_T && !dead; ++i) {
        for (int w = warp - n_prod; w < n_prod; w += n_fwd) {
            {   // record i of producer w is ready when phase i / kRfRing of its slot's barrier has completed; every lane
                // waits for itself (acquire), suspended by the hardware between the time-limited tries
                unsigned long long *bar = rf_bar + (size_t)w * kRfRing + (i % kRfRing);
                const unsigned parity = (unsigned)(i / kRfRing) & 1u;
                int tries = 0;
                while (!rf_mbar_try_wait(bar, parity)) {
                    if ((++tries & 63) == 0 && (clock64() - t0 > timeout || *(volatile int *)p.err_flag)) {
                        atomicExch(p.err_flag, 1);
                        dead = true;
                        break;
                    }
                }
            }
            dead = __any_sync(0xffffffffu, dead);
            if (dead) break;
            const double2 v = rf_ring[((size_t)w * kRfRing + (i % kRfRing)) * 32 + lane];
            __syncwarp();
            if (lane == 0) st_release_cta_shared(rf_prog + wpc + w, i + 1);
            const size_t off = ((size_t)(bw_lo + (p.rf_pack ? cta * p.rf_pack + w : w * nCTA + cta)) * (N_T + 1) + (N_T - i)) * 32 + lane;
#pragma unroll
            for (int r = 0; r < kMaxRanks; ++r)
                if (r < world) Xr[r][off] = v;  // peers over NVLink
        }
    }
}

// Rank barrier behind the backward sweep: every rank's chi trajectory is complete on every rank before anybody reads it.
// Writers: fence -> arrival (gpu-scope release); warp 0 of CTA 0 collects the arrivals of this rank, fences at system
// scope and raises this rank's flag on every rank; everybody waits for all flags in its own memory.
template <int LPT>
static __device__ __noinline__ void rf_rank_barrier(const WarpParams *pp, const int cta, const int warp, const int lane,
                                                    const int gbar) {
    const WarpParams &p = *pp;
    const int nthr = p.wpc * LPT;  // the trajectory threads of the CTA; warps without work sleep in this hardware barrier
    __threadfence_system();
    bar_sync(15, nthr);
    if (warp == 0 && lane == 0) {
        asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(p.rf_count) : "memory");
        const long long t0 = clock64();
        if (cta == 0) {
            const unsigned total = (unsigned)p.nCTA;
            unsigned seen;
            do {
                asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(p.rf_count) : "memory");
            } while (seen < total && clock64() - t0 < p.timeout_cycles);
            __threadfence_system();
            for (int r = 0; r < p.rf_world; ++r)
                asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p.rf_flag[r] + p.rf_rank), "l"(p.rf_iter) : "memory");
        }
        for (int r = 0; r < p.rf_world; ++r) {
            unsigned long long f;
            do {
                asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(f) : "l"(p.rf_flag[p.rf_rank] + r) : "memory");
                if (clock64() - t0 > p.timeout_cycles || *(volatile int *)p.err_flag) {
                    atomicExch(p.err_flag, 1);
                    break;
                }
            } while (f < p.rf_iter);
        }
        __threadfence_system();
        if (cta == 0) *reinterpret_cast<long long *>(p.err_flag + 2) = clock64() - t0;  // krotov_info.ms_rank_wait
    }
    bar_sync(15, nthr);
}

// Producer side of the replicated forward sweep's backward shard (RF instances only; empty otherwise).
template <bool RF>
struct RfProducer {};
template <>
struct RfProducer<true> {
    double2 *v0, *ring;
    unsigned long long *bar;  // [kRfRing] "record ready" barriers of this producer's slots
    int *cons;
    size_t xoff;
    int item, consumed;
    bool use_fwd, rf;
    __device__ __forceinline__ void init(double2 *plain, double2 *ring_, unsigned long long *bar_, int *cons_, size_t xoff_,
                                         bool use_fwd_, bool rf_) {
        v0 = plain; ring = ring_; bar = bar_; cons = cons_; xoff = xoff_; item = 0; consumed = 0; use_fwd = use_fwd_; rf = rf_;
    }
    // the consumer's progress, read a step ahead of its use.  A relaxed load: an acquire load puts a MEMBAR behind it that
    // waits for the metadata prefetches of the next step (their latency is otherwise hidden behind the Chebyshev terms);
    // the ring slot is only rewritten after this value has been tested (control dependency), and the forwarder
    // publishes it behind a release once its own read of the slot has been performed
    __device__ __forceinline__ void peek() {
        if (use_fwd) consumed = *reinterpret_cast<volatile int *>(cons);
    }
    template <int LPT>
    __device__ __forceinline__ void put(const WarpParams &p, const int slot, const double2 v, const int lane, const int gbar) {
        if (use_fwd) {
            while (item - consumed >= kRfRing && *(volatile int *)p.err_flag == 0) consumed = *reinterpret_cast<volatile int *>(cons);
            v0 = ring + (item % kRfRing) * 32;
            v0[lane] = v;
            __syncwarp();
            if (lane == 0) rf_mbar_arrive(bar + (item % kRfRing));  // "record `item` is in its slot" (release)
            ++item;
        } else {
            v0[lane] = v;
            grp_sync<LPT>(gbar);
            if (rf) {
                for (int r = 0; r < p.rf_world; ++r) p.Xr[r][xoff + (size_t)slot * LPT] = v;  // peers over NVLink
            } else {
                p.X[xoff + (size_t)slot * LPT] = v;
            }
        }
    }
};

// RF: instance with the replicated forward sweep of several ranks compiled in (sharded backward sweep, forwarder warps, rank
// barrier); the regular instances carry none of it (at 254 registers per thread every extra live value costs the sweeps).
// TAYLOR: the step is taylor_step (prop_method=Expmv; WarpParams::m_f / m_b then hold (m, s) pairs) instead of cheby_step.
template <int W, int LT /*0 = runtime L, rows reloaded from L1/L2 per use*/, int MAXTHREADS, int LPT = 32, bool EMUL = false,
          bool RF = false, bool TAYLOR = false>
__global__ void __launch_bounds__(MAXTHREADS, 1) krotov_warp_kernel(const __grid_constant__ WarpParams p0) {
    using Step = Prop<TAYLOR>;
    const WarpParams &p = select_params<EMUL>(p0);
    const int cta = EMUL ? (int)blockIdx.x - p.cta_base : (int)blockIdx.x;
    constexpr bool PREG = (LT > 0);
    constexpr int NT = PREG ? (1 + LT) : 1;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    // trajectory threads: `warp` = index of the trajectory group in the CTA, `lane` = row within the group;
    // the communication warp is the last 32 threads of the CTA
    const bool is_comm = (int)threadIdx.x >= p.wpc * LPT;
    const int lane = is_comm ? ((int)threadIdx.x - p.wpc * LPT) : ((int)threadIdx.x % LPT);
    const int warp = (int)threadIdx.x / LPT;
    const int gbar = 3 + warp;  // named barrier of this group (LPT > 32)
    const int L = PREG ? LT : p.L;
    const int wpc = p.wpc, tpw = p.tpw;
    // smem carve-up
    double2 *vbuf = reinterpret_cast<double2 *>(smem_raw);        // [wpc][2][LPT]
    double2 *psis = vbuf + (size_t)wpc * 2 * LPT;                 // [wpc][tpw][LPT]
    double *red = reinterpret_cast<double *>(psis + (size_t)wpc * tpw * LPT);  // [L][wpc*LPT]
    double *eps_s = red + (size_t)L * wpc * LPT;                  // [kMaxCtrl]
    double *gbuf = eps_s + kMaxCtrl;                              // [kMaxCtrl * 160] reducer scratch (CTA 0)
    double2 *chibufs = reinterpret_cast<double2 *>(gbuf + kMaxCtrl * 160);  // [wpc][LPT] chi(t_{n+1}) for the precompute
    double2 *rf_ring = chibufs + (size_t)wpc * LPT;               // [wpc][kRfRing][32]  (only with p.rf_fwd)
    unsigned long long *rf_bar = reinterpret_cast<unsigned long long *>(rf_ring + (size_t)wpc * kRfRing * 32);  // [wpc][kRfRing]
    int *rf_prog = reinterpret_cast<int *>(rf_bar + (size_t)wpc * kRfRing);  // [wpc] (unused), [wpc] records consumed
    const int nthr_all = wpc * LPT + 32;
    const int N_T = p.N_T;
    const bool rf_fwd = RF && LPT == 32 && p.rf_world > 1 && p.rf_fwd != 0 && p.mode == 1;
    if (rf_fwd) {  // (uniform over the CTA)
        if ((int)threadIdx.x < 2 * wpc) rf_prog[threadIdx.x] = 0;
        if ((int)threadIdx.x < wpc * kRfRing) rf_mbar_init(rf_bar + threadIdx.x, 1);
        __syncthreads();
    }

    if constexpr (RF) {
        if (is_comm) return;  // (the RF instances run the backward sweep only: nothing to exchange)
    }
    if (is_comm) {
        __shared__ __align__(16) WarpParams p_sh;
        comm_warp_run(p, cta, L, lane, wpc * (LPT / 32), nthr_all, red, eps_s, gbuf, &p_sh);
        return;
    }

    // -------------------------------------------------------------------- trajectory warps
    const int gw = cta * wpc + warp;       // global trajectory-warp index
    const int kbase = gw * tpw;                   // first trajectory of this warp
    double2 *bufA = vbuf + (size_t)warp * 2 * LPT;
    double2 *bufB = bufA + LPT;
    double2 *mypsi = psis + (size_t)warp * tpw * LPT;

    int col[W];
#pragma unroll
    for (int s = 0; s < W; ++s) col[s] = p.cols[s * LPT + lane];

    const size_t rowstride = (size_t)(W + 1) * LPT;   // one term
    double2 P[NT][W + 1];                            // PREG: per-term rows of this lane's trajectory
    double2 g[W + 1];

    const long long t_begin = clock64();
    long long t_wait_b = 0, t_overlap = 0, t_step = 0;
    // ================================================================ backward sweep
    const bool rf = RF && p.rf_world > 1;
    // replicated forward sweep: warps [0, n_prod) of this CTA propagate a trajectory of the backward shard, the others
    // forward the chi records to all ranks
    const int n_prod = !rf ? 0
                       : p.rf_pack ? min(p.rf_pack, max(0, p.bw_hi - p.bw_lo - cta * p.rf_pack))
                                   : min(wpc, max(0, (p.bw_hi - p.bw_lo - cta + p.nCTA - 1) / p.nCTA));
    const int n_fwd = wpc - n_prod;
    const bool use_fwd = rf_fwd && n_prod > 0 && n_fwd > 0;
    const int vw = RF ? (warp * max(1, p.rf_stride)) % wpc : warp;  // role slot of this warp
    if constexpr (RF)
        if (p.mode == 1 && use_fwd && vw >= n_prod) rf_forward_records(&p, rf_ring, rf_bar, rf_prog, cta, vw, lane, n_prod, n_fwd);
    if (p.mode == 1 && (RF || !p.skip_bw)) {
        for (int t = 0; t < tpw; ++t) {
            int k = kbase + t;
            if constexpr (RF) if (rf) {  // (tpw == 1) this rank's backward shard, spread over the CTAs: one trajectory per SM first
                const int tl = p.rf_pack ? (vw < p.rf_pack ? cta * p.rf_pack + vw : p.N) : vw * p.nCTA + cta;
                k = (tl < p.bw_hi - p.bw_lo) ? p.bw_lo + tl : p.N;
            }
            if (k >= p.N) break;
            const int gi = p.gen_of_traj[k];
            const double2 *Pg = p.Pb + (size_t)gi * (1 + L) * rowstride;
            if (PREG) {
#pragma unroll
                for (int q = 0; q < NT; ++q) load_row<W, LPT>(Pg + q * rowstride, P[q], lane);
            }
            double2 chi;
            if (p.chiT != nullptr) {
                chi = p.chiT[(size_t)k * LPT + lane];
            } else {
                const double2 c = p.chi_coef[k];
                const double2 tg = p.target[(size_t)k * LPT + lane];
                chi = make_double2(c.x * tg.x - c.y * tg.y, c.x * tg.y + c.y * tg.x);
            }
            double2 *Xk = p.X + (size_t)k * (N_T + 1) * LPT;
            // RF instances: the record goes to every rank (peer stores over NVLink) -- or, with forwarder warps, into this
            // warp's ring slot (which doubles as the next step's v_0 buffer), published with one release store; a
            // forwarder warp then stores it to every rank.  (Kept in a type that is EMPTY in the regular instances: a mere
            // unused lambda here changed their register allocation and cost the forward sweep 2 %.)
            RfProducer<RF> rfp;
            if constexpr (RF) rfp.init(mypsi + t * LPT, rf_ring + (size_t)vw * kRfRing * 32, rf_bar + (size_t)vw * kRfRing, rf_prog + wpc + vw,
                                       (size_t)k * (N_T + 1) * LPT + lane, use_fwd, rf);
            if constexpr (RF) {
                rfp.template put<LPT>(p, N_T, chi, lane, gbar);
            } else {
                Xk[(size_t)N_T * LPT + lane] = chi;
                mypsi[t * LPT + lane] = chi;
                grp_sync<LPT>(gbar);
            }
            typename Step::Meta meta = Step::load(p.dtc_b, p.m_b, p.phase_b, p.coef_b, p.ndtc_b, p.mmax_b, gi, N_T - 1);
            double e_cur[kMaxCtrl];
#pragma unroll
            for (int l = 0; l < kMaxCtrl; ++l) e_cur[l] = (l < L) ? p.amp_old[(size_t)l * N_T + N_T - 1] : 0.0;
            for (int n = N_T - 1; n >= 0; --n) {
                const int nn = n > 0 ? n - 1 : 0;  // prefetch the next step's metadata and pulse values
                const typename Step::Meta meta_next = Step::load(p.dtc_b, p.m_b, p.phase_b, p.coef_b, p.ndtc_b, p.mmax_b, gi, nn);
                double e_next[kMaxCtrl];
#pragma unroll
                for (int l = 0; l < kMaxCtrl; ++l) e_next[l] = (l < L) ? p.amp_old[(size_t)l * N_T + nn] : 0.0;
                if (PREG) {
#pragma unroll
                    for (int s = 0; s <= W; ++s) g[s] = P[0][s];
#pragma unroll
                    for (int l = 0; l < NT - 1; ++l) {
                        const double e = e_cur[l];
#pragma unroll
                        for (int s = 0; s <= W; ++s) {
                            g[s].x = fma(e, P[l + 1][s].x, g[s].x);
                            g[s].y = fma(e, P[l + 1][s].y, g[s].y);
                        }
                    }
                } else {
                    load_row<W, LPT>(Pg, g, lane);
                    for (int l = 0; l < L; ++l) {
                        const double e = p.amp_old[(size_t)l * N_T + n];  // (runtime index: reload, L1 hit)
                        const double2 *Pl = Pg + (size_t)(l + 1) * rowstride;
#pragma unroll
                        for (int s = 0; s <= W; ++s) {
                            const double2 v = Pl[s * LPT + lane];
                            g[s].x = fma(e, v.x, g[s].x);
                            g[s].y = fma(e, v.y, g[s].y);
                        }
                    }
                }
                if constexpr (RF) {
                    rfp.peek();  // (consumer's progress: used when the next record is put)
                    chi = Step::template step<W, LPT>(chi, g, col, rfp.v0, bufA, bufB, meta, lane, gbar);
                } else {
                    chi = Step::template step<W, LPT>(chi, g, col, mypsi + t * LPT, bufA, bufB, meta, lane, gbar);
                }
                meta = meta_next;
#pragma unroll
                for (int l = 0; l < kMaxCtrl; ++l) e_cur[l] = e_next[l];
                if constexpr (RF) {
                    rfp.template put<LPT>(p, n, chi, lane, gbar);
                } else {
                    mypsi[t * LPT + lane] = chi;
                    grp_sync<LPT>(gbar);
                    Xk[(size_t)n * LPT + lane] = chi;
                }
            }
        }
        if constexpr (RF)
            if (rf) rf_rank_barrier<LPT>(&p, cta, warp, lane, gbar);
    }
    if constexpr (RF) {
        // Stage 1 of the replicated forward sweep ends here; the forward sweep is a launch of the REGULAR instance
        // (skip_bw = 1).  Compiled together with the forward sweep, this backward sweep ran 0.15-0.3 us per time step
        // behind the regular one (register allocation of the bigger function).
        if (p.prof != nullptr && warp == 0 && lane == 0) p.prof[cta * 8 + 0] = clock64() - t_begin;
        return;
    }

    const long long t_bw_end = clock64();
    // ================================================================ forward sweep
    double2 psi_reg = make_double2(0.0, 0.0);
    for (int t = 0; t < tpw; ++t) {
        const int k = kbase + t;
        double2 v = make_double2(0.0, 0.0);
        if (k < p.N) {
            v = p.psi0[(size_t)k * LPT + lane];
            if (p.store_fw) p.Phi[(size_t)k * (N_T + 1) * LPT + lane] = v;
        }
        mypsi[t * LPT + lane] = v;
        if (t == 0) psi_reg = v;
    }
    grp_sync<LPT>(gbar);
    const int k0 = kbase;
    const int g0 = (k0 < p.N) ? p.gen_of_traj[k0] : 0;
    if (PREG && k0 < p.N) {
        const double2 *Pg = p.Pf + (size_t)g0 * (1 + L) * rowstride;
#pragma unroll
        for (int q = 0; q < NT; ++q) load_row<W, LPT>(Pg + q * rowstride, P[q], lane);
    }
    const double inv_s0 = (k0 < p.N) ? p.inv_s_f[g0] : 0.0;
    typename Step::Meta fmeta = Step::load(p.dtc_f, p.m_f, p.phase_f, p.coef_f, p.ndtc_f, p.mmax_f, g0, 0);
    double2 chi_next = make_double2(0.0, 0.0);
    if (p.mode == 1 && k0 < p.N) chi_next = p.X[(size_t)k0 * (N_T + 1) * LPT + lane];
    // FAST: register-resident rows, one trajectory per warp, Hermitian control terms.  Then
    //   Im<chi|mu_l|psi> = -(1/s) Re <P_l chi|psi>   (P_l = -i s mu_l is anti-Hermitian)
    // so xi_l = P_l chi(t_n) can be formed BEFORE psi(t_n) exists, and the overlap on the critical path is a
    // plain dot product; and the products w_t = P_t psi(t_n) that make up the first Chebyshev term
    // v_1 = (w_0 + sum_l eps_l w_l) / 2 are formed while the warp waits for eps.
    const bool FAST = !TAYLOR && PREG && tpw == 1 && p.mode == 1 && p.mu_hermitian != 0;
    double2 *chibuf = chibufs + (size_t)warp * LPT;
    double2 xi[PREG ? (LT > 0 ? LT : 1) : 1];
    double2 wv[PREG ? NT : 1];
    if (PREG && FAST) {
        chibuf[lane] = chi_next;
        grp_sync<LPT>(gbar);
#pragma unroll
        for (int l = 0; l < NT - 1; ++l) {
            double wr = 0.0, wi = 0.0;
            row_dot<W>(P[l + 1], col, chibuf, chi_next, wr, wi);
            xi[l] = make_double2(wr, wi);
        }
        grp_sync<LPT>(gbar);
    }

    for (int n = 0; n < N_T; ++n) {
        double eps[PREG ? (LT > 0 ? LT : 1) : kMaxCtrl];
        const long long ts0 = clock64();
        if (p.mode == 1) {
            // ---- overlaps  Im <chi_k| mu_l |psi_k>   (src/optimize.jl:339-349)
            double part[PREG ? (LT > 0 ? LT : 1) : kMaxCtrl];
#pragma unroll
            for (int l = 0; l < (PREG ? LT : kMaxCtrl); ++l) part[l] = 0.0;
            if (PREG && FAST) {
                if (k0 < p.N) {
#pragma unroll
                    for (int l = 0; l < NT - 1; ++l)
                        part[l] = -inv_s0 * fma(xi[l].x, psi_reg.x, xi[l].y * psi_reg.y);
                }
            } else
            for (int t = 0; t < tpw; ++t) {
                const int k = kbase + t;
                if (k >= p.N) break;
                const int gi = (t == 0) ? g0 : p.gen_of_traj[k];
                const double inv_s = (t == 0) ? inv_s0 : p.inv_s_f[gi];
                const double2 psi = (tpw == 1) ? psi_reg : mypsi[t * LPT + lane];
                const double2 chi = (t == 0) ? chi_next : p.X[((size_t)k * (N_T + 1) + n) * LPT + lane];
                if (PREG) {
#pragma unroll
                    for (int l = 0; l < NT - 1; ++l) {
                        double wr = 0.0, wi = 0.0;
                        row_dot<W>(P[l + 1], col, mypsi + t * LPT, psi, wr, wi);
                        part[l] = fma(inv_s, fma(chi.x, wr, chi.y * wi), part[l]);
                    }
                } else {
                    const double2 *Pg = p.Pf + (size_t)gi * (1 + L) * rowstride;
                    for (int l = 0; l < L; ++l) {
                        load_row<W, LPT>(Pg + (size_t)(l + 1) * rowstride, g, lane);
                        double wr = 0.0, wi = 0.0;
                        row_dot<W>(g, col, mypsi + t * LPT, psi, wr, wi);
                        part[l] = fma(inv_s, fma(chi.x, wr, chi.y * wi), part[l]);
                    }
                }
            }
#pragma unroll
            for (int l = 0; l < (PREG ? LT : kMaxCtrl); ++l)
                if (l < L) red[(size_t)l * wpc * LPT + warp * LPT + lane] = part[l];
            bar_arrive(1, nthr_all);  // barrier A
            const long long w0 = clock64();
            t_overlap += w0 - ts0;
            if (n + 1 < N_T && k0 < p.N) chi_next = p.X[((size_t)k0 * (N_T + 1) + n + 1) * LPT + lane];
            if (PREG && FAST && k0 < p.N) {
                // ---- idle window: everything for this and the next step that does not depend on eps_n
#pragma unroll
                for (int q = 0; q < NT; ++q) {
                    double wr = 0.0, wi = 0.0;
                    row_dot<W>(P[q], col, mypsi, psi_reg, wr, wi);
                    wv[q] = make_double2(wr, wi);
                }
                chibuf[lane] = chi_next;
                grp_sync<LPT>(gbar);
#pragma unroll
                for (int l = 0; l < NT - 1; ++l) {
                    double wr = 0.0, wi = 0.0;
                    row_dot<W>(P[l + 1], col, chibuf, chi_next, wr, wi);
                    xi[l] = make_double2(wr, wi);
                }
                grp_sync<LPT>(gbar);
            }
            bar_sync(2, nthr_all);    // barrier B: updated pulse value is in eps_s
#pragma unroll
            for (int l = 0; l < (PREG ? LT : kMaxCtrl); ++l)
                if (l < L) eps[l] = eps_s[l];
            if (p.prof != nullptr) {  // the barrier is deferred-blocking: time the wait at the first consumer
                asm volatile("" ::"d"(eps[0]) : "memory");
                t_wait_b += clock64() - w0;
            }
        } else {
#pragma unroll
            for (int l = 0; l < (PREG ? LT : kMaxCtrl); ++l)
                if (l < L) eps[l] = p.amp_old[(size_t)l * N_T + n];
        }
        // ---- forward step with the (updated) pulse value  (src/optimize.jl:360-368)
        const typename Step::Meta fmeta_next =
            Step::load(p.dtc_f, p.m_f, p.phase_f, p.coef_f, p.ndtc_f, p.mmax_f, g0, n + 1 < N_T ? n + 1 : n);
        for (int t = 0; t < tpw; ++t) {
            const int k = kbase + t;
            if (k >= p.N) break;
            const int gi = (t == 0) ? g0 : p.gen_of_traj[k];
            const typename Step::Meta sm = (t == 0) ? fmeta : Step::load(p.dtc_f, p.m_f, p.phase_f, p.coef_f, p.ndtc_f, p.mmax_f, gi, n);
            if (PREG) {
#pragma unroll
                for (int s = 0; s <= W; ++s) g[s] = P[0][s];
#pragma unroll
                for (int l = 0; l < NT - 1; ++l) {
#pragma unroll
                    for (int s = 0; s <= W; ++s) {
                        g[s].x = fma(eps[l], P[l + 1][s].x, g[s].x);
                        g[s].y = fma(eps[l], P[l + 1][s].y, g[s].y);
                    }
                }
            } else {
                const double2 *Pg = p.Pf + (size_t)gi * (1 + L) * rowstride;
                load_row<W, LPT>(Pg, g, lane);
                for (int l = 0; l < L; ++l) {
                    const double2 *Pl = Pg + (size_t)(l + 1) * rowstride;
#pragma unroll
                    for (int s = 0; s <= W; ++s) {
                        const double2 v = Pl[s * LPT + lane];
                        g[s].x = fma(eps[l], v.x, g[s].x);
                        g[s].y = fma(eps[l], v.y, g[s].y);
                    }
                }
            }
            double2 psi = (tpw == 1) ? psi_reg : mypsi[t * LPT + lane];
            if (PREG && FAST) {  // (never in the TAYLOR instances)
                double v1r = wv[0].x, v1i = wv[0].y;
#pragma unroll
                for (int l = 0; l < NT - 1; ++l) {
                    v1r = fma(eps[l], wv[l + 1].x, v1r);
                    v1i = fma(eps[l], wv[l + 1].y, v1i);
                }
                psi = cheby_step_from_v1<W, LPT>(psi, make_double2(0.5 * v1r, 0.5 * v1i), g, col, bufA, bufB, sm.a, sm.m,
                                            sm.phase, lane, gbar);
            } else {
                psi = Step::template step<W, LPT>(psi, g, col, mypsi + t * LPT, bufA, bufB, sm, lane, gbar);
            }
            mypsi[t * LPT + lane] = psi;
            if (t == 0) psi_reg = psi;
            grp_sync<LPT>(gbar);
            if (p.store_fw) {
                // mode 1 writes slot n like the reference (sic, src/optimize.jl:367); the plain
                // forward sweep writes slot n+1 (src/optimize.jl:263)
                const int slot = (p.mode == 1) ? n : n + 1;
                p.Phi[((size_t)k * (N_T + 1) + slot) * LPT + lane] = psi;
            }
        }
        fmeta = fmeta_next;
        if (p.prof != nullptr) {
            asm volatile("" ::"d"(psi_reg.x) : "memory");
            t_step += clock64() - ts0;
        }
    }

    if (p.prof != nullptr && warp == 0 && lane == 0) {
        const long long t_end = clock64();
        if (!p.skip_bw) p.prof[cta * 8 + 0] = t_bw_end - t_begin;
        p.prof[cta * 8 + 1] = t_end - t_bw_end;
        p.prof[cta * 8 + 2] = t_wait_b;
        p.prof[cta * 8 + 6] = t_overlap;
        p.prof[cta * 8 + 7] = t_step;
    }
    // ---- final states and tau_k = <tgt_k|psi_k(T)>  (src/optimize.jl:378-381)
    for (int t = 0; t < tpw; ++t) {
        const int k = kbase + t;
        if (k >= p.N) break;
        const double2 psi = mypsi[t * LPT + lane];
        p.psi_final[(size_t)k * LPT + lane] = psi;
        double tr = 0.0, ti = 0.0;
        if (p.target != nullptr) {
            const double2 tg = p.target[(size_t)k * LPT + lane];
            tr = tg.x * psi.x + tg.y * psi.y;
            ti = tg.x * psi.y - tg.y * psi.x;
        }
        tr = warp_sum_xor(tr);
        ti = warp_sum_xor(ti);
        if (LPT > 32) {  // combine the group's warps through its (now free) Chebyshev buffer
            grp_sync<LPT>(gbar);
            if ((lane & 31) == 0) bufA[lane >> 5] = make_double2(tr, ti);
            grp_sync<LPT>(gbar);
            tr = 0.0;
            ti = 0.0;
            for (int q = 0; q < LPT / 32; ++q) {
                tr += bufA[q].x;
                ti += bufA[q].y;
            }
        }
        if (lane == 0) p.tau[k] = make_double2(tr, ti);
    }
}

}  // namespace kr
