// Dense-generator engine: the batched Chebyshev propagator as FP64 tensor-core complex GEMMs (sm_100a).
//
// For Hilbert spaces too large for the warp-per-trajectory kernel the trajectories that share a generator
// are propagated TOGETHER: the state block Psi is a (d x N) complex matrix and every Chebyshev term
//     V_j = G V_{j-1} + V_{j-2},      G = 2c (H_0 - beta + sum_l eps_l[n] H_l)   (d x d, dense)
// is one complex GEMM with a fused epilogue (recursion, running sum  OUT += a_j V_j, and on the last term the
// phase e^{-i beta dt}, the store of chi(t_n) into the HBM trajectory and nothing else).  The GEMM runs on the
// FP64 tensor pipe: `mma.sync.m8n8k4.f64` (DMMA; tcgen05 has no FP64 kind).  Complex arithmetic is the 4M form
//     C_r += G_r X_r + (-G_i) X_i,    C_i += G_r X_i + G_i X_r
// on interleaved (re, im) operands: one 16-byte shared-memory load feeds the real and the imaginary fragment.
//
// Kernel shape: CTA tile 32 rows x up to 64 trajectories; 4 consumer warps (one 8-row DMMA tile each, all
// column tiles: 32 accumulator registers pairs) + 1 producer warp that streams K-chunks of 32 through a
// 4-stage shared-memory ring with bulk async copies (`cp.async.bulk` -> SASS UBLKCP) completing on mbarriers.
// Rows are padded in shared memory (A: 36, X: 66 sixteen-byte words per row) so that the DMMA fragment loads
// of every quarter-warp hit 8 different bank groups.
//
// Time-serial forward sweep without host round trips: per time step the host only ENQUEUES kernels
//   overlap GEMMs (H_l Psi, epilogue reduces Im<chi|H_l|psi> per CTA) -> update kernel (fixed-order sum,
//   pulse update written to device memory) -> build-G kernel (reads the new pulse value from device memory)
//   -> m-1 GEMMs;
// the pulse value never visits the host.
#include "dense_kernel.cuh"
#include "device_buffer.cuh"

#include <cooperative_groups.h>

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>

namespace kr {

using cplx = std::complex<double>;

namespace {

constexpr int BM = 32;       // rows per CTA
constexpr int BK = 32;       // complex k per stage
constexpr int STAGES = 4;
constexpr int A_STRIDE = 36;  // 16-byte words per A row in smem (32 + 4 pad)
constexpr int X_STRIDE = 66;  // 16-byte words per X row in smem (64 + 2 pad)
constexpr int A_STAGE_WORDS = BM * A_STRIDE;
constexpr int X_STAGE_WORDS = BK * X_STRIDE;
constexpr int STAGE_WORDS = A_STAGE_WORDS + X_STAGE_WORDS;
constexpr int GEMM_THREADS = 160;
constexpr int kMaxL = 8;

#define DK_CHECK(call)                                                                 \
    do {                                                                               \
        cudaError_t e_ = (call);                                                       \
        if (e_ != cudaSuccess) {                                                       \
            err = std::string(#call) + ": " + cudaGetErrorString(e_);                  \
            return false;                                                              \
        }                                                                              \
    } while (0)

// ---------------------------------------------------------------- PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void dmma(double &c0, double &c1, const double a, const double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

struct GemmParams {
    const double2 *A;   // [dp][dp] row-major
    const double2 *B;   // [dp][ld] row-major state block, columns col0 .. col0 + 8*NT
    int dp, ld, col0;
    int epi;            // 0 = Chebyshev term, 1 = overlap partial sums
    // ---- epi 0
    const double2 *Vold;  // V_{j-2}  (j == 1: unused)
    double2 *Vnew;        // V_j
    double2 *OUT;         // running sum
    int j, last;
    double a0, aj;
    double2 phase;
    double2 *PSI;         // last term: phase * OUT
    double2 *store;       // last term: optional second copy (storage slot), same layout
    // ---- epi 1
    const double2 *CHI;
    double *partial;      // [dp / BM] one entry per row block
    // ---- operand staging: ONE bulk copy per tile when the operand is tile-contiguous in global memory
    int a_tiled;          // A is stored tile-major [row block][k chunk][BM][A_STRIDE] (the per-step generator G)
    int x_contig;         // ld == 8 NT + 2: the BK rows of a B tile are one contiguous piece (single column block)
    // ---- stream-K (grid = SM count > row blocks): partial tiles and their ready flags
    int streamk;
    double2 *ws;          // [dp / BM][kSkParts][BM * 64]
    unsigned *flags;      // [dp / BM][kSkParts][4]: 1 = partial tile parked; the owner resets it to 0 after reading
};

constexpr int kSkParts = 8;  // most CTAs that can share one row block

__device__ __forceinline__ void st_release_u32(unsigned *p, unsigned v) {
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned *p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// CTA c of a stream-K launch owns the chunks [total * c / G, total * (c + 1) / G) of the linearised (row block, k chunk)
// space; this is the CTA that owns chunk x.
__device__ __forceinline__ int sk_cta_of(long long x, long long total, int G) {
    int c = (int)((x * G) / total);
    while (c + 1 < G && total * (c + 1) / G <= x) ++c;
    while (c > 0 && total * c / G > x) --c;
    return c;
}

template <int NT>
__global__ void __launch_bounds__(GEMM_THREADS, 1) dense_gemm_kernel(const __grid_constant__ GemmParams p) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double2 *ring = reinterpret_cast<double2 *>(smem_raw);
    uint64_t *full = reinterpret_cast<uint64_t *>(ring + (size_t)STAGES * STAGE_WORDS);
    uint64_t *empty = full + STAGES;
    double *wsum = reinterpret_cast<double *>(empty + STAGES);  // [4] per-warp partials (epi 1)
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nk = p.dp / BK;
    constexpr uint32_t X_ROW_BYTES = NT * 8 * 16;
    // shared-memory row stride of the B tile: the global leading dimension when the tile arrives in one piece
    const int xs = p.x_contig ? NT * 8 + 2 : X_STRIDE;
    const uint32_t a_bytes = p.a_tiled ? BM * A_STRIDE * 16 : BM * BK * 16;
    const uint32_t x_bytes = p.x_contig ? BK * (NT * 8 + 2) * 16 : BK * X_ROW_BYTES;
    const uint32_t STAGE_BYTES = a_bytes + x_bytes;
    // Work of this CTA: a contiguous range of (row block, k chunk) pairs.  Classic launch: one whole row block.
    // Stream-K launch (as many CTAs as SMs, more than row blocks): total / G chunks each, so a row block is shared by
    // the CTAs whose ranges meet inside it.  The CTA that holds a row block's LAST chunk owns it: it adds the partial
    // tiles of the others (fixed order: ascending k) and runs the epilogue.  A CTA works on its trailing partial
    // segment FIRST and on the segment it owns last, so nobody ever waits on a CTA that is itself waiting.
    const long long total = (long long)(p.dp / BM) * nk;
    const int G = gridDim.x;
    const long long lo = p.streamk ? total * blockIdx.x / G : (long long)blockIdx.x * nk;
    const long long hi = p.streamk ? total * (blockIdx.x + 1) / G : lo + nk;
    const int rb_first = (int)(lo / nk), rb_last = (int)((hi - 1) / nk);
    const int nseg = rb_last - rb_first + 1;
    const bool tail_first = (hi % nk) != 0 && nseg > 1;  // trailing segment does not finish its row block

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 4);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    // segment q of this CTA in processing order
    auto segment = [&](int q, int &rb, int &k0, int &k1) {
        int idx = q;
        if (tail_first) idx = (q == 0) ? nseg - 1 : q - 1;
        rb = rb_first + idx;
        k0 = (rb == rb_first) ? (int)(lo - (long long)rb_first * nk) : 0;
        k1 = (rb == rb_last) ? (int)(hi - (long long)rb_last * nk) : nk;
    };

    if (warp == 4) {
        // ------------------------------------------------------------ producer: bulk copies, one row per lane
        int it = 0;
        for (int q = 0; q < nseg; ++q) {
            int rb, k0, k1;
            segment(q, rb, k0, k1);
            const int row0 = rb * BM;
            for (int kc = k0; kc < k1; ++kc, ++it) {
                const int s = it % STAGES;
                if (it >= STAGES) mbar_wait(&empty[s], ((it / STAGES) - 1) & 1);
                double2 *As = ring + (size_t)s * STAGE_WORDS;
                double2 *Xs = As + A_STAGE_WORDS;
                if (lane == 0) mbar_expect_tx(&full[s], STAGE_BYTES);
                __syncwarp();
                // a bulk copy costs the copy engine ~50 cycles whatever its size: 64 row-sized copies per stage kept
                // the GEMM at 1.2 TB/s of generator however few columns it had; tile-contiguous operands need two
                if (p.a_tiled) {
                    if (lane == 0) bulk_g2s(As, p.A + ((size_t)rb * nk + kc) * (BM * A_STRIDE), a_bytes, &full[s]);
                } else {
                    bulk_g2s(As + lane * A_STRIDE, p.A + (size_t)(row0 + lane) * p.dp + (size_t)kc * BK, BK * 16, &full[s]);
                }
                if (p.x_contig) {
                    if (lane == 1) bulk_g2s(Xs, p.B + (size_t)(kc * BK) * p.ld, x_bytes, &full[s]);
                } else {
                    bulk_g2s(Xs + lane * X_STRIDE, p.B + (size_t)(kc * BK + lane) * p.ld + p.col0, X_ROW_BYTES, &full[s]);
                }
            }
        }
        return;
    }

    // ---------------------------------------------------------------- consumers: DMMA
    const int fr = lane >> 2, fk = lane & 3;  // fragment row / k (A), fragment col / k (B)
    int it = 0;
    for (int q = 0; q < nseg; ++q) {
        int rb, k0, k1;
        segment(q, rb, k0, k1);
        const int row0 = rb * BM;
        double cr[NT][2], ci[NT][2];
#pragma unroll
        for (int t = 0; t < NT; ++t) cr[t][0] = cr[t][1] = ci[t][0] = ci[t][1] = 0.0;
        for (int kc = k0; kc < k1; ++kc, ++it) {
            const int s = it % STAGES;
            mbar_wait(&full[s], (it / STAGES) & 1);
            const double2 *As = ring + (size_t)s * STAGE_WORDS + (warp * 8 + fr) * A_STRIDE + fk;
            const double2 *Xs = ring + (size_t)s * STAGE_WORDS + A_STAGE_WORDS + fk * xs + fr;
#pragma unroll
            for (int ks = 0; ks < BK / 4; ++ks) {
                const double2 a = As[ks * 4];
                const double nai = -a.y;
                // two passes over the column tiles: the two DMMAs that feed one accumulator are 2 NT - 1 instructions
                // apart instead of back to back (the asm statements are volatile: this IS the issue order)
                double2 x[NT];
#pragma unroll
                for (int t = 0; t < NT; ++t) x[t] = Xs[(ks * 4) * xs + t * 8];
#pragma unroll
                for (int t = 0; t < NT; ++t) {
                    dmma(cr[t][0], cr[t][1], a.x, x[t].x);
                    dmma(ci[t][0], ci[t][1], a.x, x[t].y);
                }
#pragma unroll
                for (int t = 0; t < NT; ++t) {
                    dmma(cr[t][0], cr[t][1], nai, x[t].y);
                    dmma(ci[t][0], ci[t][1], a.y, x[t].x);
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[s]);
        }

        if (p.streamk && (k0 > 0 || k1 < nk)) {
            const int first_cta = sk_cta_of((long long)rb * nk, total, G);
            const int slot = (int)blockIdx.x - first_cta;  // position among the CTAs sharing this row block
            if (k1 < nk) {
                // ---- contributor: park the partial tile, raise the flag of this warp's 8 rows
                double2 *wt = p.ws + ((size_t)rb * kSkParts + slot) * (BM * 64) + (size_t)(warp * 8 + fr) * (NT * 8) + 2 * fk;
#pragma unroll
                for (int t = 0; t < NT; ++t) {
                    wt[t * 8] = make_double2(cr[t][0], ci[t][0]);
                    wt[t * 8 + 1] = make_double2(cr[t][1], ci[t][1]);
                }
                __syncwarp();
                if (lane == 0) st_release_u32(p.flags + ((size_t)rb * kSkParts + slot) * 4 + warp, 1u);
                continue;
            }
            // ---- owner: add the partial tiles of the CTAs before this one, ascending k
            double sr[NT][2], si[NT][2];
#pragma unroll
            for (int t = 0; t < NT; ++t) sr[t][0] = sr[t][1] = si[t][0] = si[t][1] = 0.0;
            for (int sl = 0; sl < slot; ++sl) {
                unsigned *fl = p.flags + ((size_t)rb * kSkParts + sl) * 4 + warp;
                if (lane == 0)
                    while (ld_acquire_u32(fl) != 1u) {
                    }
                __syncwarp();
                const double2 *wt = p.ws + ((size_t)rb * kSkParts + sl) * (BM * 64) + (size_t)(warp * 8 + fr) * (NT * 8) + 2 * fk;
#pragma unroll
                for (int t = 0; t < NT; ++t) {
                    const double2 u0 = __ldcg(wt + t * 8), u1 = __ldcg(wt + t * 8 + 1);
                    sr[t][0] += u0.x; si[t][0] += u0.y;
                    sr[t][1] += u1.x; si[t][1] += u1.y;
                }
                __syncwarp();
                if (lane == 0) *fl = 0u;  // consumed: the next launch (stream-ordered, or a graph replay) starts clean
            }
#pragma unroll
            for (int t = 0; t < NT; ++t) {
                cr[t][0] = sr[t][0] + cr[t][0]; ci[t][0] = si[t][0] + ci[t][0];
                cr[t][1] = sr[t][1] + cr[t][1]; ci[t][1] = si[t][1] + ci[t][1];
            }
        }

        // ---------------------------------------------------------------- epilogue of a finished row block
        const int row = row0 + warp * 8 + fr;
        if (p.epi == 0) {
#pragma unroll
            for (int t = 0; t < NT; ++t) {
                const size_t idx = (size_t)row * p.ld + p.col0 + t * 8 + 2 * fk;
                double2 v0, v1, o0, o1;
                if (p.j == 1) {
                    const double2 b0 = p.B[idx], b1 = p.B[idx + 1];  // V_0
                    v0 = make_double2(0.5 * cr[t][0], 0.5 * ci[t][0]);
                    v1 = make_double2(0.5 * cr[t][1], 0.5 * ci[t][1]);
                    o0 = make_double2(fma(p.aj, v0.x, p.a0 * b0.x), fma(p.aj, v0.y, p.a0 * b0.y));
                    o1 = make_double2(fma(p.aj, v1.x, p.a0 * b1.x), fma(p.aj, v1.y, p.a0 * b1.y));
                } else {
                    const double2 w0 = p.Vold[idx], w1 = p.Vold[idx + 1];
                    const double2 q0 = p.OUT[idx], q1 = p.OUT[idx + 1];
                    v0 = make_double2(cr[t][0] + w0.x, ci[t][0] + w0.y);
                    v1 = make_double2(cr[t][1] + w1.x, ci[t][1] + w1.y);
                    o0 = make_double2(fma(p.aj, v0.x, q0.x), fma(p.aj, v0.y, q0.y));
                    o1 = make_double2(fma(p.aj, v1.x, q1.x), fma(p.aj, v1.y, q1.y));
                }
                if (p.last) {
                    const double2 r0 = make_double2(p.phase.x * o0.x - p.phase.y * o0.y, p.phase.x * o0.y + p.phase.y * o0.x);
                    const double2 r1 = make_double2(p.phase.x * o1.x - p.phase.y * o1.y, p.phase.x * o1.y + p.phase.y * o1.x);
                    p.PSI[idx] = r0;
                    p.PSI[idx + 1] = r1;
                    if (p.store) {
                        p.store[idx] = r0;
                        p.store[idx + 1] = r1;
                    }
                } else {
                    p.Vnew[idx] = v0;
                    p.Vnew[idx + 1] = v1;
                    p.OUT[idx] = o0;
                    p.OUT[idx + 1] = o1;
                }
            }
        } else {
            // Im <chi | w> = chi_r w_i - chi_i w_r, summed over the row block's tile in a fixed order
            double acc = 0.0;
#pragma unroll
            for (int t = 0; t < NT; ++t) {
                const size_t idx = (size_t)row * p.ld + p.col0 + t * 8 + 2 * fk;
                const double2 c0 = p.CHI[idx], c1 = p.CHI[idx + 1];
                acc += c0.x * ci[t][0] - c0.y * cr[t][0];
                acc += c1.x * ci[t][1] - c1.y * cr[t][1];
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
            asm volatile("bar.sync 1, 128;" ::: "memory");  // wsum of the previous segment has been read
            if (lane == 0) wsum[warp] = acc;
            asm volatile("bar.sync 1, 128;" ::: "memory");  // the 4 consumer warps only
            if (warp == 0 && lane == 0) p.partial[rb] = (wsum[0] + wsum[1]) + (wsum[2] + wsum[3]);
        }
    }
}

// G = f (H_0 - beta + sum_l eps_l[n] H_l)   elementwise; eps is read from DEVICE memory (no host round trip)
__global__ void build_G_kernel(double2 *G, const double2 *H, int dp, int L, double2 f, double beta, const double *eps,
                               int N_T, int n) {
    const size_t total = (size_t)dp * dp;
    double e[kMaxL];
    for (int l = 0; l < L; ++l) e[l] = eps[(size_t)l * N_T + n];
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        double2 h = H[i];
        const size_t r = i / dp, c = i - r * dp;
        if (r == c) h.x -= beta;
        for (int l = 0; l < L; ++l) {
            const double2 hl = H[(size_t)(l + 1) * total + i];
            h.x = fma(e[l], hl.x, h.x);
            h.y = fma(e[l], hl.y, h.y);
        }
        // tile-major [row block][k chunk][BM][A_STRIDE]: exactly the shared-memory image of a GEMM stage
        const size_t dst = ((r / BM) * (size_t)(dp / BK) + c / BK) * (BM * A_STRIDE) + (r % BM) * A_STRIDE + (c % BK);
        G[dst] = make_double2(f.x * h.x - f.y * h.y, f.x * h.y + f.y * h.x);
    }
}

// x = tanh(s_l e) for a saturating control (bounded amplitudes), else e.  Out of line: the persistent sweeps that
// inline amp_apply keep their register allocation whether or not saturation is in use.
static __device__ __noinline__ double amp_saturate(const double *sat, const int l, const double e) {
    return sat[l] != 0.0 ? tanh(sat[l] * e) : e;
}

// coefficient of H_l in the generator for the control value e (non-linear amplitudes, src/optimize.jl:268-272)
__device__ __forceinline__ double amp_apply(const AmpDev &am, const int l, const int N_T, const int n, double e) {
    if (am.sat != nullptr) e = amp_saturate(am.sat, l, e);
    double c = e;
    if (am.poly != nullptr) {
        const double *q = am.poly + l * (kAmpDeg + 1);
        c = q[kAmpDeg];
#pragma unroll
        for (int d = kAmpDeg - 1; d >= 0; --d) c = fma(c, e, q[d]);
    }
    if (am.shape != nullptr) c = __dmul_rn(am.shape[(size_t)l * N_T + n], c);
    return c;
}

// Tied control terms (krotov_set_control_terms), one thread, once the overlap sums s[t] of every term are known over all
// ranks: term t moves with du of its control, the sum over the control's terms in ascending t of a_t'(eps_old) s[t]
// (src/optimize.jl:351-358 with mu = sum_t a_t' H_t).  On return s[t] = a_t(eps_new), the coefficient of H_t in the
// forward step; eps_new and ga are written when `write`.  Out of line: the sweeps keep their code for untied problems.
// P: the launch parameters (update_kernel's arguments, SweepParams or DSweepParams), read through a pointer to the
// grid constant.
template <class P>
static __device__ __noinline__ void tie_update_cold(const P *pp, const int n, double *s, const bool write) {
    const P &p = *pp;
    const int L = p.L, N_T = p.N_T;
    const double *ctrl = p.am.tie, *dfac = p.am.tie + L;
    double du[kMaxL];
    for (int t = 0; t < L; ++t) {
        bool first = true;
        for (int u = 0; u < L; ++u)
            if (ctrl[u] == ctrl[t]) {
                const double v = __dmul_rn(dfac[(size_t)u * N_T + n], s[u]);
                du[t] = first ? v : __dadd_rn(du[t], v);
                first = false;
            }
    }
    for (int t = 0; t < L; ++t) {
        const double a = p.alpha[(size_t)t * N_T + n];
        const double e_new = __dadd_rn(p.eps_old[(size_t)t * N_T + n], __dmul_rn(a, du[t]));  // :355-356
        s[t] = amp_apply(p.am, t, N_T, n, e_new);
        if (write) {
            p.eps_new[(size_t)t * N_T + n] = e_new;
            const double prev = (n == 0) ? 0.0 : p.ga[t];
            p.ga[t] = __dadd_rn(prev, __dmul_rn(__dmul_rn(a, __dmul_rn(fabs(du[t]), fabs(du[t]))), p.dt[n]));  // :357
        }
    }
}

// update_kernel's arguments in the shape tie_update_cold reads
struct UpdateArgs {
    int L, N_T;
    const double *alpha, *eps_old, *dt;
    double *eps_new, *ga;
    AmpDev am;
};

// The rank's sum `s` of control l at time step n -> the sum over all ranks, the same bits on every rank: the rank sum is
// pushed into slot [rank] of every rank's mailbox (system-scope stores over NVLink, by the caller flagged `push` only)
// and the `world` slots of the own mailbox are polled and added in rank order.  Called by ONE lane; every CTA of the
// persistent sweeps calls it (they all need the total), the pushing is done by CTA 0.
__device__ __forceinline__ double rank_sum_lane(const DenseComm &cm, const int L, const int n, const int l, const double s,
                                                const bool push) {
    if (cm.world <= 1) return s;
    const size_t off = ((size_t)n * L + l) * cm.world;
    if (push)
        for (int r = 0; r < cm.world; ++r)
            asm volatile("st.relaxed.sys.global.f64 [%0], %1;" ::"l"(cm.mbox[r] + off + cm.rank), "d"(s) : "memory");
    double tot = 0.0;
    const long long t0 = clock64();
    for (int r = 0; r < cm.world; ++r) {
        unsigned long long u;
        int spins = 0;
        for (;;) {
            asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(u) : "l"(cm.mbox[cm.rank] + off + r) : "memory");
            if (u != 0xFFFFFFFFFFFFFFFFull) break;
            if ((++spins & 63) == 0 && (clock64() - t0 > cm.timeout_cycles || *(volatile int *)cm.err_flag)) {
                atomicExch(cm.err_flag, 1);
                break;
            }
        }
        tot += __longlong_as_double((long long)u);
    }
    return tot;
}

// fixed-order sum of the CTA partials of control term l and the rank exchange; every lane returns the sum.
// With several ranks the rank sum is pushed into every peer's mailbox (system-scope stores over NVLink) and
// the `world` slots are summed in rank order -- the same protocol as the warp path's reducer.
__device__ __forceinline__ double term_sum(const double *partial, const int n_partial, const int L, const int l, const int n,
                                           const DenseComm &cm, const int lane) {
    double s = 0.0;
    for (int c = lane; c < n_partial; c += 32) s += partial[(size_t)l * n_partial + c];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (cm.world > 1) {
        const size_t off = ((size_t)n * L + l) * cm.world;
        if (lane < cm.world)
            asm volatile("st.relaxed.sys.global.f64 [%0], %1;" ::"l"(cm.mbox[lane] + off + cm.rank), "d"(s) : "memory");
        const double *mine = cm.mbox[cm.rank] + off + (lane < cm.world ? lane : 0);
        unsigned long long u;
        const long long t0 = clock64();
        int spins = 0;
        for (;;) {
            asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(u) : "l"(mine) : "memory");
            if (__all_sync(0xffffffffu, u != 0xFFFFFFFFFFFFFFFFull)) break;
            if ((++spins & 63) == 0 && (clock64() - t0 > cm.timeout_cycles || *(volatile int *)cm.err_flag)) {
                atomicExch(cm.err_flag, 1);
                break;
            }
        }
        const double v = __longlong_as_double((long long)u);
        s = 0.0;
        for (int r = 0; r < cm.world; ++r) s += __shfl_sync(0xffffffffu, v, r);
    }
    return s;
}

// pulse update (src/optimize.jl:351-358): block l updates term l
__global__ void update_kernel(const double *partial, int n_partial, int L, const double *alpha, const double *eps_old,
                              double *eps_new, double *ga, const double *dt, int N_T, int n, DenseComm cm, AmpDev am) {
    const int l = blockIdx.x, lane = threadIdx.x;
    double s = term_sum(partial, n_partial, L, l, n, cm, lane);
    if (lane == 0) {
        const double a = alpha[(size_t)l * N_T + n];
        if (am.dfac != nullptr) s = __dmul_rn(am.dfac[(size_t)l * N_T + n], s);  // mu_l = a_l'(eps^(i)) H_l
        const double e_new = __dadd_rn(eps_old[(size_t)l * N_T + n], __dmul_rn(a, s));
        eps_new[(size_t)l * N_T + n] = e_new;
        if (am.amp_new != nullptr) am.amp_new[(size_t)l * N_T + n] = amp_apply(am, l, N_T, n, e_new);
        const double prev = (n == 0) ? 0.0 : ga[l];
        ga[l] = __dadd_rn(prev, __dmul_rn(__dmul_rn(a, __dmul_rn(fabs(s), fabs(s))), dt[n]));
    }
}

// the same for tied control terms: ONE block sums every term, then ties them (tie_update_cold)
__global__ void update_tied_kernel(const double *partial, int n_partial, int L, const double *alpha, const double *eps_old,
                                   double *eps_new, double *ga, const double *dt, int N_T, int n, DenseComm cm, AmpDev am) {
    __shared__ double s_sh[kMaxL];
    const int lane = threadIdx.x;
    for (int t = 0; t < L; ++t) {
        const double s = term_sum(partial, n_partial, L, t, n, cm, lane);
        if (lane == 0) s_sh[t] = s;
    }
    if (lane == 0) {
        const UpdateArgs u{L, N_T, alpha, eps_old, dt, eps_new, ga, am};
        tie_update_cold(&u, n, s_sh, true);
        for (int t = 0; t < L; ++t) am.amp_new[(size_t)t * N_T + n] = s_sh[t];
    }
}

// tau_k = <tgt_k | psi_k>: one warp per column
__global__ void tau_kernel(const double2 *PSI, const double2 *TGT, int d, int ld, const int *col_of_traj, int N,
                           double2 *tau) {
    const int k = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (k >= N) return;
    const int c = col_of_traj[k];
    double tr = 0.0, ti = 0.0;
    for (int i = lane; i < d; i += 32) {
        const double2 t = TGT[(size_t)i * ld + c], x = PSI[(size_t)i * ld + c];
        tr += t.x * x.x + t.y * x.y;
        ti += t.x * x.y - t.y * x.x;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        tr += __shfl_xor_sync(0xffffffffu, tr, o);
        ti += __shfl_xor_sync(0xffffffffu, ti, o);
    }
    if (lane == 0) tau[k] = make_double2(tr, ti);
}

// chi(T)[i][col] = coef[k] * tgt[i][col]
__global__ void chi_from_coef_kernel(double2 *CHI, const double2 *TGT, const double2 *coef, const int *traj_of_col,
                                     int dp, int ld) {
    const size_t total = (size_t)dp * ld;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % ld);
        const int k = traj_of_col[c];
        double2 out = make_double2(0.0, 0.0);
        if (k >= 0) {
            const double2 a = coef[k], t = TGT[i];
            out = make_double2(a.x * t.x - a.y * t.y, a.x * t.y + a.y * t.x);
        }
        CHI[i] = out;
    }
}

// ============================================================================ sparse generators, d > 32
// The same block propagator for SPARSE generators (spin chains, coupled-oscillator networks ...): the Chebyshev
// term is an SpMM over the state block.  ELL storage with one shared pattern: slot 0 of every row is the
// diagonal, `cols[row][s]` / values `[row][s]`; padded slots point at the own row with value 0.  One warp owns 4
// rows x 32 trajectories: the generator entry is a warp-uniform (broadcast) load, the gathered state row is one
// coalesced 512-byte read served by L1/L2 (the state blocks of all terms fit the 126 MB L2), so the kernel is
// bound by L2 -> SM bandwidth, not by FP64.  Same fused epilogues as the dense GEMM.
constexpr int SP_ROWS_PER_WARP = 4;
constexpr int SP_WARPS = 8;
constexpr int SP_ROWS = SP_ROWS_PER_WARP * SP_WARPS;

struct SpmmParams {
    const int *cols;      // [dp][W]
    const double2 *Gv;    // [dp][W]
    int W, ncols;         // ELL width; columns of this block (multiple of 8)
    GemmParams e;         // B, dp, ld, col0 and the epilogue fields
};

__device__ __forceinline__ void cheby_epilogue_1(const GemmParams &p, const size_t idx, const double cr, const double ci) {
    double2 v, o;
    if (p.j == 1) {
        const double2 b0 = p.B[idx];
        v = make_double2(0.5 * cr, 0.5 * ci);
        o = make_double2(fma(p.aj, v.x, p.a0 * b0.x), fma(p.aj, v.y, p.a0 * b0.y));
    } else {
        const double2 w0 = p.Vold[idx], q0 = p.OUT[idx];
        v = make_double2(cr + w0.x, ci + w0.y);
        o = make_double2(fma(p.aj, v.x, q0.x), fma(p.aj, v.y, q0.y));
    }
    if (p.last) {
        const double2 r = make_double2(p.phase.x * o.x - p.phase.y * o.y, p.phase.x * o.y + p.phase.y * o.x);
        p.PSI[idx] = r;
        if (p.store) p.store[idx] = r;
    } else {
        p.Vnew[idx] = v;
        p.OUT[idx] = o;
    }
}

__global__ void __launch_bounds__(SP_WARPS * 32) spmm_kernel(const __grid_constant__ SpmmParams p) {
    __shared__ double wsum[SP_WARPS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c = blockIdx.y * 32 + lane;
    const bool cvalid = c < p.ncols;
    const int row0 = blockIdx.x * SP_ROWS + warp * SP_ROWS_PER_WARP;
    const GemmParams &e = p.e;
    double cr[SP_ROWS_PER_WARP], ci[SP_ROWS_PER_WARP], cr1[SP_ROWS_PER_WARP], ci1[SP_ROWS_PER_WARP];
#pragma unroll
    for (int q = 0; q < SP_ROWS_PER_WARP; ++q) cr[q] = ci[q] = cr1[q] = ci1[q] = 0.0;
    const size_t cbase = (size_t)e.col0 + (cvalid ? c : 0);
    // The gathers are latency-bound (ncu: long-scoreboard stalls dominate), so 4 slots x 4 rows = 16 independent
    // state-row loads are put in flight before the first FMA.
    constexpr int SU = 4;
    int s = 0;
    for (; s + SU <= p.W; s += SU) {
        int jj[SU][SP_ROWS_PER_WARP];
        double2 gg[SU][SP_ROWS_PER_WARP], xx[SU][SP_ROWS_PER_WARP];
#pragma unroll
        for (int u = 0; u < SU; ++u)
#pragma unroll
            for (int q = 0; q < SP_ROWS_PER_WARP; ++q) {
                const size_t slot = (size_t)(row0 + q) * p.W + s + u;
                jj[u][q] = p.cols[slot];  // warp-uniform
                gg[u][q] = p.Gv[slot];    // warp-uniform
            }
#pragma unroll
        for (int u = 0; u < SU; ++u)
#pragma unroll
            for (int q = 0; q < SP_ROWS_PER_WARP; ++q) xx[u][q] = e.B[(size_t)jj[u][q] * e.ld + cbase];
#pragma unroll
        for (int u = 0; u < SU; ++u)
#pragma unroll
            for (int q = 0; q < SP_ROWS_PER_WARP; ++q) {
                cr[q] = fma(gg[u][q].x, xx[u][q].x, cr[q]);
                cr1[q] = fma(-gg[u][q].y, xx[u][q].y, cr1[q]);
                ci[q] = fma(gg[u][q].x, xx[u][q].y, ci[q]);
                ci1[q] = fma(gg[u][q].y, xx[u][q].x, ci1[q]);
            }
    }
    for (; s < p.W; ++s) {
#pragma unroll
        for (int q = 0; q < SP_ROWS_PER_WARP; ++q) {
            const size_t slot = (size_t)(row0 + q) * p.W + s;
            const int j = p.cols[slot];
            const double2 g = p.Gv[slot];
            const double2 x = e.B[(size_t)j * e.ld + cbase];
            cr[q] = fma(g.x, x.x, cr[q]);
            cr1[q] = fma(-g.y, x.y, cr1[q]);
            ci[q] = fma(g.x, x.y, ci[q]);
            ci1[q] = fma(g.y, x.x, ci1[q]);
        }
    }
    if (e.epi == 0) {
        if (cvalid) {
#pragma unroll
            for (int q = 0; q < SP_ROWS_PER_WARP; ++q)
                cheby_epilogue_1(e, (size_t)(row0 + q) * e.ld + cbase, cr[q] + cr1[q], ci[q] + ci1[q]);
        }
    } else {
        double acc = 0.0;
        if (cvalid) {
#pragma unroll
            for (int q = 0; q < SP_ROWS_PER_WARP; ++q) {
                const double2 ch = e.CHI[(size_t)(row0 + q) * e.ld + cbase];
                acc += ch.x * (ci[q] + ci1[q]) - ch.y * (cr[q] + cr1[q]);
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) wsum[warp] = acc;
        __syncthreads();
        if (threadIdx.x == 0) {
            double t = 0.0;
            for (int w = 0; w < SP_WARPS; ++w) t += wsum[w];
            e.partial[blockIdx.y * gridDim.x + blockIdx.x] = t;
        }
    }
}

// ELL values of G = f (P_0 - beta on the diagonal slot + sum_l eps_l[n] P_l); eps read from device memory
__global__ void build_G_sparse_kernel(double2 *Gv, const double2 *Pv, size_t nslots, int W, int L, double2 f,
                                      double beta, const double *eps, int N_T, int n) {
    double ev[kMaxL];
    for (int l = 0; l < L; ++l) ev[l] = eps[(size_t)l * N_T + n];
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nslots; i += (size_t)gridDim.x * blockDim.x) {
        double2 h = Pv[i];
        if (i % W == 0) h.x -= beta;  // slot 0 is the diagonal
        for (int l = 0; l < L; ++l) {
            const double2 hl = Pv[(size_t)(l + 1) * nslots + i];
            h.x = fma(ev[l], hl.x, h.x);
            h.y = fma(ev[l], hl.y, h.y);
        }
        Gv[i] = make_double2(f.x * h.x - f.y * h.y, f.x * h.y + f.y * h.x);
    }
}

// ============================================================================ persistent sweep, sparse generators
// The launch-per-term stream above costs ~14 us per Chebyshev term on mid-sized problems whose SpMM takes 3-6 us
// (profiles/r1_sparse_vs_dense.txt: 10 spins, d = 1024: 265 us per time step for 19 launches).  This kernel runs a
// whole Krotov iteration (or the plain forward sweep) of the sparse path in ONE cooperative launch: every warp owns
// a fixed set of (4 rows x 32 columns) items for the whole sweep, builds the generator values of its rows once per
// time step from the pulse values into shared memory (no build_G pass, no G in global memory), and the Chebyshev
// terms are separated by grid barriers (the only thing a term needs from other CTAs is V_{j-1}).  The per-step
// overlap sums go through one more barrier: CTA partials, then every CTA adds them in the same fixed order, so all
// CTAs hold the same new pulse value without a broadcast.  Same state blocks, storage and arithmetic per element as
// spmm_kernel / build_G_sparse_kernel / update_kernel (the overlap sums differ in summation order only).
struct SweepParams {
    int dp, ld, W, L, N_T, n_blocks, n_items, mode, store_fw, K;  // K = items per warp (shared-memory slots)
    int cg_sync;               // 1 = cooperative-groups grid.sync() instead of the counter barrier
    unsigned *bar;             // barrier counter (zeroed before the launch)
    const int *cols;           // [dp][W]
    const double2 *Pv[2];      // per direction: [g][1+L][dp*W]
    const int *blk;            // [n_blocks][4]: generator, first column, columns, first item
    const double *coef[2];     // [g][ndtc][mmax]
    const int *m[2];           // [g][ndtc]
    const double2 *phase[2];   // [g][ndtc]
    const int *dtc[2];         // [N_T]
    const double *E_min[2], *Delta[2];  // [g]
    int ndtc[2], mmax[2];
    double2 *PSI, *V[3], *OUT, *X, *PHI;
    const double2 *PSI0, *CHI;
    size_t slab;
    const double *eps_old, *alpha, *dt;
    double *eps_new, *ga;
    double *partial;           // [L][gridDim.x]
    const double *amp_old;     // a(eps_old): coefficients of the generator under the known pulses (== eps_old when linear)
    AmpDev am;
    DenseComm cm;              // several ranks: mailboxes of this iteration's parity
};

struct SweepItem {
    int b, g, row0, ncols, c;  // column block, generator, first row, columns of the block, this lane's column
    size_t cbase;
    bool valid, cvalid;
};

template <int R>
__device__ __forceinline__ SweepItem sweep_item(const SweepParams &p, const int it, const int lane) {
    SweepItem r;
    r.valid = it < p.n_items;
    int b = 0;
    if (r.valid)
        while (b + 1 < p.n_blocks && p.blk[(b + 1) * 4 + 3] <= it) ++b;
    r.b = b;
    r.g = p.blk[b * 4 + 0];
    r.ncols = p.blk[b * 4 + 2];
    const int local = r.valid ? it - p.blk[b * 4 + 3] : 0;
    const int rgs = p.dp / R;
    const int cg_ = local / rgs;
    r.row0 = (local - cg_ * rgs) * R;
    r.c = cg_ * 32 + lane;
    r.cvalid = r.valid && r.c < r.ncols;
    r.cbase = (size_t)p.blk[b * 4 + 1] + (r.cvalid ? r.c : 0);
    return r;
}

// rows of G (or of a control term) times the state block B for one item: the same loop as spmm_kernel, generator
// values and column indices from this warp's shared-memory copy
template <int R>
__device__ __forceinline__ void sweep_rows_times_block(const double2 *__restrict__ gv, const int *__restrict__ cl, const int W,
                                                       const double2 *B /* rewritten during the launch: no .nc loads */, const int ld, const size_t cbase,
                                                       double (&outr)[R], double (&outi)[R]) {
    double cr[R], ci[R], cr1[R], ci1[R];
#pragma unroll
    for (int q = 0; q < R; ++q) cr[q] = ci[q] = cr1[q] = ci1[q] = 0.0;
    constexpr int SU = 16 / R;  // 16 state-row loads in flight per lane
    int s = 0;
    for (; s + SU <= W; s += SU) {
        double2 gg[SU][R], xx[SU][R];
#pragma unroll
        for (int u = 0; u < SU; ++u)
#pragma unroll
            for (int q = 0; q < R; ++q) {
                gg[u][q] = gv[q * W + s + u];
                xx[u][q] = B[(size_t)cl[q * W + s + u] * ld + cbase];
            }
#pragma unroll
        for (int u = 0; u < SU; ++u)
#pragma unroll
            for (int q = 0; q < R; ++q) {
                cr[q] = fma(gg[u][q].x, xx[u][q].x, cr[q]);
                cr1[q] = fma(-gg[u][q].y, xx[u][q].y, cr1[q]);
                ci[q] = fma(gg[u][q].x, xx[u][q].y, ci[q]);
                ci1[q] = fma(gg[u][q].y, xx[u][q].x, ci1[q]);
            }
    }
    for (; s < W; ++s) {
#pragma unroll
        for (int q = 0; q < R; ++q) {
            const double2 g = gv[q * W + s];
            const double2 x = B[(size_t)cl[q * W + s] * ld + cbase];
            cr[q] = fma(g.x, x.x, cr[q]);
            cr1[q] = fma(-g.y, x.y, cr1[q]);
            ci[q] = fma(g.x, x.y, ci[q]);
            ci1[q] = fma(g.y, x.x, ci1[q]);
        }
    }
#pragma unroll
    for (int q = 0; q < R; ++q) {
        outr[q] = cr[q] + cr1[q];
        outi[q] = ci[q] + ci1[q];
    }
}

// Grid barrier: one monotonic counter; thread 0 of every CTA arrives (release) and spins (acquire), bar.sync on both
// sides extends the ordering to the whole CTA (the pattern of cooperative groups' grid.sync, without its bookkeeping).
__device__ __forceinline__ void sweep_barrier(const SweepParams &p, cooperative_groups::grid_group &grid, unsigned &target) {
    if (p.cg_sync) {
        grid.sync();
        return;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        target += gridDim.x;
        __threadfence();
        asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(p.bar) : "memory");
        while ((int)(ld_acquire_u32(p.bar) - target) < 0) {
        }
        __threadfence();
    }
    __syncthreads();
}

// One propagation step of the whole state block: m_step - 1 terms, a grid barrier behind each.
template <int R>
__device__ __forceinline__ void sweep_step(const SweepParams &p, cooperative_groups::grid_group &grid, const int dir,
                                           const int n, const double (&eps)[kMaxL], double2 *store, double2 *gsm, int *csm,
                                           const int lane, const int wg, const int total_warps, unsigned &bar_target,
                                           const SweepItem &it0) {
    const int rowsz = R * p.W;
    const size_t nslots = (size_t)p.dp * p.W;
    const int dtc = p.dtc[dir][n];
    int m_step = 0;
    for (int b = 0; b < p.n_blocks; ++b) m_step = max(m_step, p.m[dir][p.blk[b * 4] * p.ndtc[dir] + dtc]);
    // generator rows of this warp's items for this time step (same arithmetic as build_G_sparse_kernel)
    for (int k = 0; k < p.K; ++k) {
        const SweepItem it = (k == 0) ? it0 : sweep_item<R>(p, wg + k * total_warps, lane);  // items never change
        if (!it.valid) break;
        const double sc = 4.0 / p.Delta[dir][it.g], beta = p.Delta[dir][it.g] / 2 + p.E_min[dir][it.g];
        const double2 f = (dir == KROTOV_FORWARD) ? make_double2(0.0, -sc) : make_double2(0.0, sc);
        const double2 *Pv = p.Pv[dir] + (size_t)it.g * (1 + p.L) * nslots + (size_t)it.row0 * p.W;
        for (int i = lane; i < rowsz; i += 32) {
            double2 h = Pv[i];
            if (i % p.W == 0) h.x -= beta;
            for (int l = 0; l < p.L; ++l) {
                const double2 hl = Pv[(size_t)(l + 1) * nslots + i];
                h.x = fma(eps[l], hl.x, h.x);
                h.y = fma(eps[l], hl.y, h.y);
            }
            gsm[k * rowsz + i] = make_double2(f.x * h.x - f.y * h.y, f.x * h.y + f.y * h.x);
        }
    }
    __syncwarp();
    // per-step metadata of the first item (the only one unless the problem outgrows the grid)
    const int ci0 = it0.g * p.ndtc[dir] + dtc;
    const int m0 = p.m[dir][ci0];
    const double2 ph0 = p.phase[dir][ci0];
    const double *a_0 = p.coef[dir] + (size_t)ci0 * p.mmax[dir];
    const double a00 = a_0[0];
    const double2 *vprev = p.PSI, *vprev2 = nullptr;
    for (int j = 1; j < m_step; ++j) {
        double2 *vnew = p.V[j % 3];
        for (int k = 0; k < p.K; ++k) {
            const SweepItem it = (k == 0) ? it0 : sweep_item<R>(p, wg + k * total_warps, lane);  // items never change
            if (!it.valid) break;
            const int ci_ = (k == 0) ? ci0 : it.g * p.ndtc[dir] + dtc;
            const int m = (k == 0) ? m0 : p.m[dir][ci_];
            if (j >= m) continue;
            // the epilogue's operands at this lane's own elements are requested before the gathers (one L2 round trip less)
            double2 w0[R], q0[R];
#pragma unroll
            for (int q = 0; q < R; ++q) {
                const size_t idx = (size_t)(it.row0 + q) * p.ld + it.cbase;
                w0[q] = (j == 1) ? vprev[idx] : vprev2[idx];
                q0[q] = (j == 1) ? make_double2(0.0, 0.0) : p.OUT[idx];
            }
            double cr[R], ci[R];
            sweep_rows_times_block<R>(gsm + k * rowsz, csm + k * rowsz, p.W, vprev, p.ld, it.cbase, cr, ci);
            if (!it.cvalid) continue;
            const double *a = (k == 0) ? a_0 : p.coef[dir] + (size_t)ci_ * p.mmax[dir];
            const double a0 = (k == 0) ? a00 : a[0], aj = a[j];
            const bool last = (j == m - 1);
            const double2 ph = (k == 0) ? ph0 : p.phase[dir][ci_];
#pragma unroll
            for (int q = 0; q < R; ++q) {
                const size_t idx = (size_t)(it.row0 + q) * p.ld + it.cbase;
                double2 v, o;
                if (j == 1) {
                    v = make_double2(0.5 * cr[q], 0.5 * ci[q]);
                    o = make_double2(fma(aj, v.x, a0 * w0[q].x), fma(aj, v.y, a0 * w0[q].y));
                } else {
                    v = make_double2(cr[q] + w0[q].x, ci[q] + w0[q].y);
                    o = make_double2(fma(aj, v.x, q0[q].x), fma(aj, v.y, q0[q].y));
                }
                if (last) {
                    const double2 r = make_double2(ph.x * o.x - ph.y * o.y, ph.x * o.y + ph.y * o.x);
                    p.PSI[idx] = r;
                    if (store) store[idx] = r;
                } else {
                    vnew[idx] = v;
                    p.OUT[idx] = o;
                }
            }
        }
        sweep_barrier(p, grid, bar_target);
        vprev2 = vprev;
        vprev = vnew;
    }
}

template <int R>
__global__ void __launch_bounds__(SP_WARPS * 32, 2) sparse_sweep_kernel(const __grid_constant__ SweepParams p) {
    cooperative_groups::grid_group grid = cooperative_groups::this_grid();
    extern __shared__ __align__(16) unsigned char sweep_smem[];
    __shared__ double wsum[kMaxL][SP_WARPS];
    __shared__ double eps_sh[kMaxL];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int wg = blockIdx.x * SP_WARPS + warp, total_warps = gridDim.x * SP_WARPS;
    const SweepItem it0 = sweep_item<R>(p, wg, lane);
    const int rowsz = R * p.W;
    double2 *gsm = reinterpret_cast<double2 *>(sweep_smem) + (size_t)warp * p.K * rowsz;
    int *csm = reinterpret_cast<int *>(reinterpret_cast<double2 *>(sweep_smem) + (size_t)SP_WARPS * p.K * rowsz) +
               (size_t)warp * p.K * rowsz;
    // column indices of this warp's rows never change
    for (int k = 0; k < p.K; ++k) {
        const SweepItem it = (k == 0) ? it0 : sweep_item<R>(p, wg + k * total_warps, lane);  // items never change
        if (!it.valid) break;
        for (int i = lane; i < rowsz; i += 32) csm[k * rowsz + i] = p.cols[(size_t)it.row0 * p.W + i];
    }
    __syncwarp();
    const size_t gtid = (size_t)blockIdx.x * blockDim.x + threadIdx.x, gthreads = (size_t)gridDim.x * blockDim.x;
    double eps[kMaxL];
#pragma unroll
    for (int l = 0; l < kMaxL; ++l) eps[l] = 0.0;
    unsigned bar_target = 0;

    if (p.mode == 1) {
        // ---- backward sweep: chi(t_n) for all n into X
        for (size_t i = gtid; i < p.slab; i += gthreads) {
            const double2 v = p.CHI[i];
            p.PSI[i] = v;
            p.X[p.slab * (size_t)p.N_T + i] = v;
        }
        sweep_barrier(p, grid, bar_target);
        for (int n = p.N_T - 1; n >= 0; --n) {
            for (int l = 0; l < p.L; ++l) eps[l] = p.amp_old[(size_t)l * p.N_T + n];
            sweep_step<R>(p, grid, KROTOV_BACKWARD, n, eps, p.X + p.slab * (size_t)n, gsm, csm, lane, wg, total_warps, bar_target, it0);
        }
    }
    // ---- forward sweep
    for (size_t i = gtid; i < p.slab; i += gthreads) {
        const double2 v = p.PSI0[i];
        p.PSI[i] = v;
        if (p.store_fw && p.mode == 0) p.PHI[i] = v;
    }
    sweep_barrier(p, grid, bar_target);
    const size_t nslots = (size_t)p.dp * p.W;
    for (int n = 0; n < p.N_T; ++n) {
        if (p.mode == 1) {
            // overlaps Im <chi_k(t_n)| mu_l |psi_k(t_n)> summed over this CTA's items (src/optimize.jl:339-349)
            const double2 *CHI = p.X + p.slab * (size_t)n;
            for (int l = 0; l < p.L; ++l) {
                double acc = 0.0;
                for (int k = 0; k < p.K; ++k) {
                    const SweepItem it = (k == 0) ? it0 : sweep_item<R>(p, wg + k * total_warps, lane);  // items never change
                    if (!it.valid) break;
                    const double2 *mu = p.Pv[0] + ((size_t)it.g * (1 + p.L) + 1 + l) * nslots + (size_t)it.row0 * p.W;
                    double cr[R], ci[R];
                    sweep_rows_times_block<R>(mu, csm + k * rowsz, p.W, p.PSI, p.ld, it.cbase, cr, ci);
                    if (it.cvalid) {
#pragma unroll
                        for (int q = 0; q < R; ++q) {
                            const double2 ch = CHI[(size_t)(it.row0 + q) * p.ld + it.cbase];
                            acc += ch.x * ci[q] - ch.y * cr[q];
                        }
                    }
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
                if (lane == 0) wsum[l][warp] = acc;
            }
            __syncthreads();
            if ((int)threadIdx.x < p.L) {
                double t = 0.0;
                for (int w = 0; w < SP_WARPS; ++w) t += wsum[threadIdx.x][w];
                p.partial[(size_t)threadIdx.x * gridDim.x + blockIdx.x] = t;
            }
            sweep_barrier(p, grid, bar_target);
            // every CTA adds the CTA partials in the same fixed order (lane-strided, then a butterfly): same bits everywhere
            if (warp == 0) {
                for (int l = 0; l < p.L; ++l) {
                    double sacc = 0.0;
                    for (int c = lane; c < (int)gridDim.x; c += 32) sacc += p.partial[(size_t)l * gridDim.x + c];
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) sacc += __shfl_xor_sync(0xffffffffu, sacc, o);
                    if (lane == 0) {
                        const double a = p.alpha[(size_t)l * p.N_T + n];
                        sacc = rank_sum_lane(p.cm, p.L, n, l, sacc, blockIdx.x == 0);
                        if (p.am.tie != nullptr) {
                            eps_sh[l] = sacc;  // tied control terms: the update waits for the sums of all terms
                        } else {
                            if (p.am.dfac != nullptr) sacc = __dmul_rn(p.am.dfac[(size_t)l * p.N_T + n], sacc);
                            const double e_new = __dadd_rn(p.eps_old[(size_t)l * p.N_T + n], __dmul_rn(a, sacc));  // :355-356
                            eps_sh[l] = amp_apply(p.am, l, p.N_T, n, e_new);
                            if (blockIdx.x == 0) {
                                p.eps_new[(size_t)l * p.N_T + n] = e_new;
                                const double prev = (n == 0) ? 0.0 : p.ga[l];
                                p.ga[l] = __dadd_rn(prev, __dmul_rn(__dmul_rn(a, __dmul_rn(fabs(sacc), fabs(sacc))), p.dt[n]));  // :357
                            }
                        }
                    }
                }
                if (p.am.tie != nullptr && lane == 0)
                    tie_update_cold(&p, n, eps_sh, blockIdx.x == 0);
            }
            __syncthreads();
            for (int l = 0; l < p.L; ++l) eps[l] = eps_sh[l];
            __syncthreads();
        } else {
            for (int l = 0; l < p.L; ++l) eps[l] = p.amp_old[(size_t)l * p.N_T + n];
        }
        double2 *store = nullptr;
        if (p.store_fw) store = p.PHI + p.slab * (size_t)(p.mode == 1 ? n : n + 1);  // slot n in an iteration (sic, :367)
        sweep_step<R>(p, grid, KROTOV_FORWARD, n, eps, store, gsm, csm, lane, wg, total_warps, bar_target, it0);
    }
}

}  // namespace
}  // namespace kr
#include "dense_sweep.cuh"
namespace kr {
namespace {

struct Block {  // one GEMM column block
    int g, col0, nt;
};

struct Cheb {
    bool set = false;
    int ndtc = 0, mmax = 0;
    std::vector<int> dtc_of_step, m;
    std::vector<double> E_min, Delta, coef;
    std::vector<cplx> phase;
};

}  // namespace

struct DenseEngine {
    int d = 0, dp = 0, N = 0, L = 0, N_T = 0, n_gen = 0, store_fw = 0, ld = 0;
    bool hermitian = true;
    cudaStream_t stream = nullptr;
    std::vector<int> col_of_traj, traj_of_col;
    std::vector<Block> blocks;
    int n_partial = 0;
    // device
    DevBuf Hf, Hb, G;                                            // double2
    DevBuf V[3], OUT, PSI, PSI0, TGT, CHI, X, PHI;               // double2
    DevBuf partial;                                              // double
    DevBuf d_col_of_traj, d_traj_of_col;                         // int
    bool chi_from_host = false;
    Cheb ch[2];
    size_t slab = 0;  // elements per time slot
    long long launches = 0;
    int sm_count = 148;
    DenseComm comm;
    AmpDev amp;
    // sparse mode (ELL): shared pattern, values per generator and term for both directions
    bool sparse = false;
    int W = 0;
    DevBuf ell_cols;      // int
    DevBuf Pvf, Pvb, Gv;  // double2: [g][1+L][dp*W], [g][dp*W]
    std::vector<int> sp_part_off;  // offset of every column block's CTA partials
    int nnz_union = 0;
    bool x_contig = false;   // single column block stored with ld = 8 nt + 2: a B tile is one bulk copy
    size_t gmat = 0;         // elements of one tile-major generator: (dp/BM) (dp/BK) BM A_STRIDE
    // stream-K GEMM (fewer row blocks than SMs): partial tiles, ready flags
    bool streamk = false;
    DevBuf sk_ws;     // double2
    DevBuf sk_flags;  // unsigned
    // whole-iteration CUDA graph (launch-bound problems): captured the second time an identical iteration is asked for
    unsigned long long cheb_version = 0;
    struct GraphKey {
        unsigned long long cheb_version = ~0ull;
        const void *ptr[8] = {};
        bool operator==(const GraphKey &o) const {
            return cheb_version == o.cheb_version && memcmp(ptr, o.ptr, sizeof(ptr)) == 0;
        }
    } graph_key, last_key;
    cudaGraphExec_t graph_exec = nullptr;
    long long graph_launches = 0, last_launches = 0;
    int stable_iterations = 0;
    long long graph_replays = 0;
    // persistent sweep (sparse path): launch shape and device copies of the small tables
    bool sweep = false;
    int sw_grid = 0, sw_K = 0, sw_items = 0, sw_R = 4;
    DevBuf sw_bar;  // unsigned
    size_t sw_smem = 0;
    DevBuf sw_blk, sw_m[2], sw_dtc[2];                       // int
    DevBuf sw_partial, sw_coef[2], sw_Emin[2], sw_Delta[2];  // double
    DevBuf sw_phase[2];                                      // double2
    long long sweep_launches = 0;
    int kernel_last = 0;  // enum krotov_kernel of the last forward/iterate call
    // persistent cluster sweep for moderate dense generators (dense_sweep.cuh)
    bool dsweep = false;
    int ds_units = 0, ds_R = 0, ds_gpad = 0;
    size_t ds_smem = 0;
    DevBuf ds_units_dev;  // int
    DevBuf ds_prof;       // long long

    ~DenseEngine() {
        if (graph_exec) cudaGraphExecDestroy(graph_exec);
    }
};

namespace {

// b holds n elements of T (at least one) afterwards
template <typename T>
bool dalloc(DevBuf &b, size_t n, std::string &err) {
    const cudaError_t e = b.allocate(std::max<size_t>(n, 1) * sizeof(T));
    if (e != cudaSuccess) {
        err = std::string("cudaMalloc of ") + std::to_string(n * sizeof(T)) + " bytes: " + cudaGetErrorString(e);
        return false;
    }
    return true;
}

size_t gemm_smem_bytes() { return (size_t)STAGES * STAGE_WORDS * 16 + 2 * STAGES * 8 + 64; }

bool launch_gemm(DenseEngine *e, const Block &b, GemmParams p, std::string &err) {
    p.dp = e->dp;
    p.ld = e->ld;
    p.col0 = b.col0;
    p.streamk = e->streamk ? 1 : 0;
    p.x_contig = e->x_contig ? 1 : 0;
    p.ws = e->sk_ws.get<double2>();
    p.flags = e->sk_flags.get<unsigned>();
    dim3 grid(e->streamk ? e->sm_count : e->dp / BM), block(GEMM_THREADS);
    const size_t smem = gemm_smem_bytes();
    static bool attr_set = false;
    if (!attr_set) {
        DK_CHECK(cudaFuncSetAttribute(dense_gemm_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        DK_CHECK(cudaFuncSetAttribute(dense_gemm_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        DK_CHECK(cudaFuncSetAttribute(dense_gemm_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        DK_CHECK(cudaFuncSetAttribute(dense_gemm_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set = true;
    }
    switch (b.nt) {
        case 1: dense_gemm_kernel<1><<<grid, block, smem, e->stream>>>(p); break;
        case 2: dense_gemm_kernel<2><<<grid, block, smem, e->stream>>>(p); break;
        case 4: dense_gemm_kernel<4><<<grid, block, smem, e->stream>>>(p); break;
        default: dense_gemm_kernel<8><<<grid, block, smem, e->stream>>>(p); break;
    }
    e->launches++;
    DK_CHECK(cudaGetLastError());
    return true;
}

bool launch_spmm(DenseEngine *e, const Block &b, const double2 *Gv, GemmParams p, int n_partial_off, std::string &err) {
    SpmmParams sp;
    memset(&sp, 0, sizeof(sp));
    p.dp = e->dp;
    p.ld = e->ld;
    p.col0 = b.col0;
    if (p.partial) p.partial += n_partial_off;
    sp.e = p;
    sp.cols = e->ell_cols.get<int>();
    sp.Gv = Gv;
    sp.W = e->W;
    sp.ncols = b.nt * 8;
    dim3 grid(e->dp / SP_ROWS, (sp.ncols + 31) / 32), block(SP_WARPS * 32);
    spmm_kernel<<<grid, block, 0, e->stream>>>(sp);
    e->launches++;
    DK_CHECK(cudaGetLastError());
    return true;
}

// Launch shape of the persistent sweep: as few items per warp as the co-resident grid allows (shared memory holds the
// generator rows and column indices of a warp's items).
const void *sweep_kernel_for(int R) {
    return R == 4 ? (const void *)sparse_sweep_kernel<4> : R == 2 ? (const void *)sparse_sweep_kernel<2> : (const void *)sparse_sweep_kernel<1>;
}

bool sweep_configure(DenseEngine *e) {
    e->sweep = false;
    if (!e->sparse) return true;
    // rows per warp item: the terms are latency-bound until the state block is large, so small problems get more,
    // shorter items.  Measured (tools/gpu_sparse_bench.py --variants, us per time step and direction, R = 4 / 2 / 1):
    // 8 spins 95.6 / 57.9 / 49.5, 10 spins 130.6 / 70.7 / 69.6, 12 spins 192.8 / 158.3 / 184.1.
    int col_groups = 0;
    for (const Block &b : e->blocks) col_groups += (b.nt * 8 + 31) / 32;
    const long long warps = (long long)e->sm_count * SP_WARPS;
    int R = 1;
    if ((long long)(e->dp / 4) * col_groups >= 4 * warps)
        R = 4;
    else if ((long long)(e->dp / 2) * col_groups >= warps)
        R = 2;
    if (const char *env = getenv("KROTOV_SWEEP_ROWS")) R = atoi(env) >= 4 ? 4 : atoi(env) >= 2 ? 2 : 1;
    e->sw_R = R;
    std::vector<int> blk;
    int items = 0;
    for (const Block &b : e->blocks) {
        blk.insert(blk.end(), {b.g, b.col0, b.nt * 8, items});
        items += (e->dp / R) * ((b.nt * 8 + 31) / 32);
    }
    e->sw_items = items;
    const size_t rowsz = (size_t)R * e->W;
    const void *fn = sweep_kernel_for(R);
    for (int K = 1; K <= 16; ++K) {
        const size_t smem = (size_t)SP_WARPS * K * rowsz * (16 + 4);
        if (smem > 200 * 1024) break;
        if (cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) break;
        int nb = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, fn, SP_WARPS * 32, smem) != cudaSuccess || nb < 1) break;
        const long long cap = (long long)nb * e->sm_count;
        if (cap * SP_WARPS * K >= items) {
            e->sw_K = K;
            e->sw_smem = smem;
            e->sw_grid = (int)std::min<long long>(cap, (items + SP_WARPS * K - 1) / (SP_WARPS * K));
            e->sweep = true;
            break;
        }
    }
    cudaGetLastError();
    if (!e->sweep) return true;
    std::string err;
    if (!dalloc<int>(e->sw_blk, blk.size(), err) || !dalloc<double>(e->sw_partial, (size_t)kMaxL * e->sw_grid, err) ||
        !dalloc<unsigned>(e->sw_bar, 1, err)) {
        e->sweep = false;
        return false;
    }
    return copy_to_device(e->sw_blk.get<int>(), blk.data(), blk.size() * 4, e->stream, true) == cudaSuccess;
}

inline const double *gen_coeffs_old(const DenseEngine *e, const double *d_eps);

// Persistent cluster sweep for moderate dense generators: one cluster of 8 CTAs per group of <= 8 columns.
bool dsweep_configure(DenseEngine *e) {
    e->dsweep = false;
    if (e->sparse || e->d > kDsMaxD || getenv("KROTOV_NO_DSWEEP")) return true;
    std::vector<int> units;
    for (const Block &b : e->blocks)
        for (int c = 0; c < b.nt * 8; c += kDsCols) {
            // columns of the block that hold a trajectory (a block is padded to a multiple of 8 columns)
            int n = 0;
            for (int q = c; q < std::min(c + kDsCols, b.nt * 8); ++q) n += (e->traj_of_col[b.col0 + q] >= 0) ? 1 : 0;
            if (n == 0) continue;
            units.insert(units.end(), {b.g, b.col0 + c, std::min(kDsCols, b.nt * 8 - c)});
        }
    const int n_units = (int)units.size() / 3;
    if (n_units == 0 || n_units * kDsCluster > e->sm_count) return true;  // all clusters must be co-resident
    e->ds_R = (e->d + kDsCluster - 1) / kDsCluster;
    e->ds_gpad = ds_stride(e->d);
    e->ds_smem = ((size_t)((e->ds_R + 7) / 8 * 8) * e->ds_gpad + (size_t)kDsCols * e->ds_gpad) * 16;
    if (e->ds_R > 8 * (kDsThreads / 32) || e->ds_smem > 220 * 1024) return true;
    if (cudaFuncSetAttribute((const void *)dense_cluster_sweep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)e->ds_smem) != cudaSuccess) {
        cudaGetLastError();
        return true;
    }
    {   // all clusters must be co-resident (they meet at a grid barrier): ask how many this device can hold
        cudaLaunchConfig_t cfg;
        memset(&cfg, 0, sizeof(cfg));
        cfg.gridDim = dim3(n_units * kDsCluster);
        cfg.blockDim = dim3(kDsThreads);
        cfg.dynamicSmemBytes = e->ds_smem;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = kDsCluster;
        at[0].val.clusterDim.y = 1;
        at[0].val.clusterDim.z = 1;
        cfg.attrs = at;
        cfg.numAttrs = 1;
        int max_clusters = 0;
        if (cudaOccupancyMaxActiveClusters(&max_clusters, dense_cluster_sweep_kernel, &cfg) != cudaSuccess ||
            max_clusters < n_units) {
            cudaGetLastError();
            return true;
        }
    }
    std::string err;
    if (!dalloc<int>(e->ds_units_dev, units.size(), err) ||
        !dalloc<double>(e->sw_partial, (size_t)kMaxL * n_units * kDsCluster, err) || !dalloc<unsigned>(e->sw_bar, 1, err))
        return false;
    if (copy_to_device(e->ds_units_dev.get<int>(), units.data(), units.size() * 4, e->stream, true) != cudaSuccess) return false;
    e->ds_units = n_units;
    e->dsweep = true;
    return true;
}

bool launch_dsweep(DenseEngine *e, int mode, const double *d_eps_old, double *d_eps_new, const double *d_alpha,
                   const double *d_dt, double *d_ga, std::string &err) {
    DSweepParams p;
    memset(&p, 0, sizeof(p));
    p.d = e->d; p.dp = e->dp; p.ld = e->ld; p.L = e->L; p.N_T = e->N_T; p.mode = mode; p.store_fw = e->store_fw;
    p.n_units = e->ds_units; p.R = e->ds_R; p.gpad = e->ds_gpad; p.units = e->ds_units_dev.get<int>();
    p.H[0] = e->Hf.get<double2>();
    p.H[1] = e->hermitian ? e->Hf.get<double2>() : e->Hb.get<double2>();
    for (int dir = 0; dir < 2; ++dir) {
        p.coef[dir] = e->sw_coef[dir].get<double>(); p.m[dir] = e->sw_m[dir].get<int>();
        p.phase[dir] = e->sw_phase[dir].get<double2>(); p.dtc[dir] = e->sw_dtc[dir].get<int>();
        p.E_min[dir] = e->sw_Emin[dir].get<double>(); p.Delta[dir] = e->sw_Delta[dir].get<double>();
        p.ndtc[dir] = e->ch[dir].ndtc; p.mmax[dir] = e->ch[dir].mmax;
    }
    p.PSI = e->PSI.get<double2>(); p.X = e->X.get<double2>(); p.PHI = e->PHI.get<double2>();
    p.VX[0] = e->V[0].get<double2>(); p.VX[1] = e->V[1].get<double2>();
    p.PSI0 = e->PSI0.get<double2>(); p.CHI = e->CHI.get<double2>(); p.slab = e->slab;
    p.eps_old = d_eps_old; p.eps_new = d_eps_new; p.alpha = d_alpha; p.dt = d_dt; p.ga = d_ga;
    p.amp_old = gen_coeffs_old(e, d_eps_old); p.am = e->amp; p.cm = e->comm;
    p.partial = e->sw_partial.get<double>();
    p.bar = e->sw_bar.get<unsigned>();
    if (getenv("KROTOV_PROF") && !e->ds_prof) dalloc<long long>(e->ds_prof, 8, err);
    p.prof = getenv("KROTOV_PROF") ? e->ds_prof.get<long long>() : nullptr;
    DK_CHECK(cudaMemsetAsync(e->sw_bar.get<unsigned>(), 0, sizeof(unsigned), e->stream));
    DK_CHECK(cudaFuncSetAttribute((const void *)dense_cluster_sweep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)e->ds_smem));
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(e->ds_units * kDsCluster);
    cfg.blockDim = dim3(kDsThreads);
    cfg.dynamicSmemBytes = e->ds_smem;
    cfg.stream = e->stream;
    cudaLaunchAttribute attrs[2];
    attrs[0].id = cudaLaunchAttributeClusterDimension;
    attrs[0].val.clusterDim.x = kDsCluster;
    attrs[0].val.clusterDim.y = 1;
    attrs[0].val.clusterDim.z = 1;
    attrs[1].id = cudaLaunchAttributeCooperative;  // all clusters co-resident: they meet at a grid barrier per time step
    attrs[1].val.cooperative = 1;
    cfg.attrs = attrs;
    cfg.numAttrs = 2;
    DK_CHECK(cudaLaunchKernelEx(&cfg, dense_cluster_sweep_kernel, p));
    e->launches++;
    e->sweep_launches++;
    if (p.prof) {  // diagnostics: where CTA 0 spent its cycles (us per time step of the sweep)
        long long h[6];
        DK_CHECK(cudaStreamSynchronize(e->stream));
        DK_CHECK(cudaMemcpy(h, e->ds_prof.get<long long>(), sizeof(h), cudaMemcpyDeviceToHost));
        const double f = 1.0 / 1965.0 / e->N_T;
        fprintf(stderr, "[dense sweep, mode %d, d=%d, %d clusters] us per time step (both sweeps of an iteration summed): "
                        "build G %.2f, tiles %.2f, exchange + cluster barrier %.2f, group reload %.2f, overlaps %.2f, "
                        "grid barrier + update %.2f\n", mode, e->d, e->ds_units, h[0] * f, h[1] * f, h[2] * f, h[3] * f,
                h[4] * f, h[5] * f);
    }
    return true;
}

// generator coefficients of a sweep under known pulses / under the updated pulses
inline const double *gen_coeffs_old(const DenseEngine *e, const double *d_eps) { return e->amp.amp_old ? e->amp.amp_old : d_eps; }
inline const double *gen_coeffs_new(const DenseEngine *e, const double *d_eps_new) { return e->amp.amp_new ? e->amp.amp_new : d_eps_new; }

bool sweep_usable(const DenseEngine *e, int mode) {
    // (several ranks: the per-step sums of the sweeps cross the ranks through the mailboxes, rank_sum_lane;
    // KROTOV_NO_SWEEP_RANKS=1 keeps the launch-per-term stream there)
    if (e->comm.world > 1 && getenv("KROTOV_NO_SWEEP_RANKS")) return false;
    return (e->sweep || e->dsweep) && e->ch[0].set && (mode == 0 || e->ch[1].set) && !getenv("KROTOV_NO_SWEEP");
}

int kernel_kind(const DenseEngine *e, int mode) {
    if (sweep_usable(e, mode)) return e->dsweep ? KROTOV_KERNEL_DENSE_SWEEP : KROTOV_KERNEL_SPARSE_SWEEP;
    return e->sparse ? KROTOV_KERNEL_SPARSE_STREAM : KROTOV_KERNEL_DMMA_STREAM;
}

template <typename T>
bool sweep_upload(DenseEngine *e, DevBuf &dst, const std::vector<T> &src, std::string &err) {
    if (!dalloc<T>(dst, src.size(), err)) return false;  // (frees the previous table first)
    DK_CHECK(copy_to_device(dst.get<void>(), src.data(), src.size() * sizeof(T), e->stream, true));
    return true;
}

bool launch_sweep(DenseEngine *e, int mode, const double *d_eps_old, double *d_eps_new, const double *d_alpha,
                  const double *d_dt, double *d_ga, std::string &err) {
    if (e->dsweep) return launch_dsweep(e, mode, d_eps_old, d_eps_new, d_alpha, d_dt, d_ga, err);
    SweepParams p;
    memset(&p, 0, sizeof(p));
    p.dp = e->dp; p.ld = e->ld; p.W = e->W; p.L = e->L; p.N_T = e->N_T; p.n_blocks = (int)e->blocks.size();
    p.n_items = e->sw_items; p.mode = mode; p.store_fw = e->store_fw; p.K = e->sw_K;
    p.cols = e->ell_cols.get<int>();
    p.Pv[0] = e->Pvf.get<double2>();
    p.Pv[1] = e->hermitian ? e->Pvf.get<double2>() : e->Pvb.get<double2>();
    p.blk = e->sw_blk.get<int>();
    for (int dir = 0; dir < 2; ++dir) {
        p.coef[dir] = e->sw_coef[dir].get<double>(); p.m[dir] = e->sw_m[dir].get<int>();
        p.phase[dir] = e->sw_phase[dir].get<double2>(); p.dtc[dir] = e->sw_dtc[dir].get<int>();
        p.E_min[dir] = e->sw_Emin[dir].get<double>(); p.Delta[dir] = e->sw_Delta[dir].get<double>();
        p.ndtc[dir] = e->ch[dir].ndtc; p.mmax[dir] = e->ch[dir].mmax;
    }
    p.PSI = e->PSI.get<double2>(); p.V[0] = e->V[0].get<double2>(); p.V[1] = e->V[1].get<double2>();
    p.V[2] = e->V[2].get<double2>(); p.OUT = e->OUT.get<double2>(); p.X = e->X.get<double2>(); p.PHI = e->PHI.get<double2>();
    p.PSI0 = e->PSI0.get<double2>(); p.CHI = e->CHI.get<double2>(); p.slab = e->slab;
    p.eps_old = d_eps_old; p.eps_new = d_eps_new; p.alpha = d_alpha; p.dt = d_dt; p.ga = d_ga;
    p.amp_old = gen_coeffs_old(e, d_eps_old); p.am = e->amp; p.cm = e->comm;
    p.partial = e->sw_partial.get<double>();
    p.cg_sync = getenv("KROTOV_SWEEP_CGSYNC") ? 1 : 0;
    p.bar = e->sw_bar.get<unsigned>();
    DK_CHECK(cudaMemsetAsync(e->sw_bar.get<unsigned>(), 0, sizeof(unsigned), e->stream));
    const void *fn = sweep_kernel_for(e->sw_R);
    DK_CHECK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)e->sw_smem));
    void *args[] = {(void *)&p};
    DK_CHECK(cudaLaunchCooperativeKernel(fn, dim3(e->sw_grid), dim3(SP_WARPS * 32), args, e->sw_smem, e->stream));
    e->launches++;
    e->sweep_launches++;
    return true;
}

// One propagation step of every column block: PSI <- exp(-/+ i H dt) PSI.   `store` = storage slot or nullptr.
bool step(DenseEngine *e, int dir, int n, const double *d_eps, double2 *store, std::string &err) {
    const Cheb &c = e->ch[dir];
    const int dtc = c.dtc_of_step[n];
    const size_t mat = (size_t)e->dp * e->dp;
    const double2 *H = (dir == KROTOV_FORWARD || e->hermitian) ? e->Hf.get<double2>() : e->Hb.get<double2>();
    const size_t nslots = (size_t)e->dp * e->W;
    for (int g = 0; g < e->n_gen; ++g) {
        const double s = 4.0 / c.Delta[g], beta = c.Delta[g] / 2 + c.E_min[g];
        const double2 f = (dir == KROTOV_FORWARD) ? make_double2(0.0, -s) : make_double2(0.0, s);
        if (e->sparse) {
            const double2 *Pv = (dir == KROTOV_FORWARD || e->hermitian) ? e->Pvf.get<double2>() : e->Pvb.get<double2>();
            build_G_sparse_kernel<<<std::max(1, (int)std::min<size_t>(e->sm_count * 4, (nslots + 255) / 256)), 256, 0,
                                    e->stream>>>(e->Gv.get<double2>() + (size_t)g * nslots, Pv + (size_t)g * (1 + e->L) * nslots,
                                                 nslots, e->W, e->L, f, beta, d_eps, e->N_T, n);
            e->launches++;
            continue;
        }
        build_G_kernel<<<e->sm_count * 4, 256, 0, e->stream>>>(e->G.get<double2>() + (size_t)g * e->gmat,
                                                             H + (size_t)g * (1 + e->L) * mat, e->dp, e->L, f, beta, d_eps,
                                                             e->N_T, n);
        e->launches++;
    }
    for (const Block &b : e->blocks) {
        const int ci = b.g * c.ndtc + dtc;
        const int m = c.m[ci];
        const double *a = &c.coef[(size_t)ci * c.mmax];
        const cplx ph = c.phase[ci];
        if (m < 2) {
            err = "Chebyshev expansion with fewer than 2 coefficients is not supported on the dense path";
            return false;
        }
        // V[0] aliases PSI for j = 1;  ring of three work blocks afterwards
        const double2 *vprev = e->PSI.get<double2>();  // V_{j-1}
        const double2 *vprev2 = nullptr;
        for (int j = 1; j < m; ++j) {
            GemmParams p;
            memset(&p, 0, sizeof(p));
            p.A = e->G.get<double2>() + (size_t)b.g * e->gmat;
            p.a_tiled = 1;
            p.B = vprev;
            p.epi = 0;
            p.Vold = vprev2;
            p.Vnew = e->V[j % 3].get<double2>();
            p.OUT = e->OUT.get<double2>();
            p.j = j;
            p.last = (j == m - 1);
            p.a0 = a[0];
            p.aj = a[j];
            p.phase = make_double2(ph.real(), ph.imag());
            // the last term must not overwrite PSI while other CTAs still read it as V_0 (only when m == 2)
            p.PSI = (m == 2) ? e->V[2].get<double2>() : e->PSI.get<double2>();
            p.store = store;
            if (e->sparse) {
                if (!launch_spmm(e, b, e->Gv.get<double2>() + (size_t)b.g * nslots, p, 0, err)) return false;
            } else if (!launch_gemm(e, b, p, err)) {
                return false;
            }
            vprev2 = vprev;
            vprev = e->V[j % 3].get<double2>();
        }
        if (m == 2) {
            err = "m == 2 on the dense path is not supported";
            return false;
        }
    }
    return true;
}

}  // namespace

DenseEngine *dense_create(int d, int N, int L, int N_T, int n_gen, const std::vector<cplx> &Hdense,
                          const std::vector<int> &gen_of_traj, const double *psi0, const double *target, int store_fw,
                          cudaStream_t stream, std::string &err, const SparseDesc *sp) {
    if (L > kMaxL) {
        err = "too many controls";
        return nullptr;
    }
    std::unique_ptr<DenseEngine> e(new DenseEngine());
    e->d = d; e->N = N; e->L = L; e->N_T = N_T; e->n_gen = n_gen; e->store_fw = store_fw; e->stream = stream;
    e->dp = (d + BM - 1) / BM * BM;
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&e->sm_count, cudaDevAttrMultiProcessorCount, dev);
    // columns: trajectories grouped by generator, groups cut into blocks of <= 64 columns (8 DMMA column tiles)
    e->col_of_traj.assign(N, -1);
    int col = 0;
    for (int g = 0; g < n_gen; ++g) {
        std::vector<int> ks;
        for (int k = 0; k < N; ++k)
            if (gen_of_traj[k] == g) ks.push_back(k);
        size_t pos = 0;
        while (pos < ks.size()) {
            const int rem = (int)std::min<size_t>(64, ks.size() - pos);
            int nt = (rem + 7) / 8;
            nt = nt <= 1 ? 1 : nt <= 2 ? 2 : nt <= 4 ? 4 : 8;
            e->blocks.push_back({g, col, nt});
            for (int i = 0; i < rem; ++i) e->col_of_traj[ks[pos + i]] = col + i;
            col += nt * 8;
            pos += rem;
        }
    }
    e->ld = col;
    // one column block (one generator, <= 64 trajectories): two pad columns make the global row stride equal to the
    // conflict-free shared-memory stride, so the BK rows of a GEMM operand tile are ONE contiguous bulk copy
    e->x_contig = sp == nullptr && e->blocks.size() == 1 && !getenv("KROTOV_NO_TILED");
    if (e->x_contig) e->ld = col + 2;
    e->gmat = (size_t)(e->dp / BM) * (e->dp / BK) * BM * A_STRIDE;
    e->traj_of_col.assign(e->ld, -1);
    for (int k = 0; k < N; ++k) e->traj_of_col[e->col_of_traj[k]] = k;
    e->slab = (size_t)e->dp * e->ld;
    e->n_partial = (int)e->blocks.size() * (e->dp / BM);
    e->sparse = (sp != nullptr);
    if (e->sparse) {
        e->W = sp->W;
        e->nnz_union = sp->nnz_union;
        e->n_partial = 0;
        for (const Block &b : e->blocks) {
            e->sp_part_off.push_back(e->n_partial);
            e->n_partial += (e->dp / SP_ROWS) * ((b.nt * 8 + 31) / 32);
        }
    }
    const size_t mat = e->sparse ? 0 : (size_t)e->dp * e->dp;
    const size_t nslots = e->sparse ? (size_t)e->dp * e->W : 0;

    // Hermitian generators: the adjoint terms are the terms themselves
    e->hermitian = e->sparse ? sp->hermitian : true;
    for (int q = 0; !e->sparse && q < n_gen * (1 + L) && e->hermitian; ++q) {
        const cplx *M = &Hdense[(size_t)q * d * d];
        for (int i = 0; i < d && e->hermitian; ++i)
            for (int j = i; j < d; ++j)
                if (M[(size_t)i * d + j] != std::conj(M[(size_t)j * d + i])) {
                    e->hermitian = false;
                    break;
                }
    }
    size_t need = (size_t)n_gen * (1 + L) * (mat + nslots) * (e->hermitian ? 1 : 2) + (size_t)n_gen * (mat + nslots);
    need += e->slab * (8 + (size_t)(N_T + 1) * (store_fw ? 2 : 1));
    size_t free_b = 0, total_b = 0;
    cudaMemGetInfo(&free_b, &total_b);
    if (need * 16 > free_b) {
        err = "dense path needs " + std::to_string(need * 16 >> 20) + " MiB of device memory, " +
              std::to_string(free_b >> 20) + " MiB free";
        return nullptr;
    }
    bool ok = dalloc<double2>(e->Hf, (size_t)n_gen * (1 + L) * mat, err) &&
              dalloc<double2>(e->G, (size_t)n_gen * e->gmat, err) && dalloc<double2>(e->V[0], e->slab, err) &&
              dalloc<double2>(e->V[1], e->slab, err) && dalloc<double2>(e->V[2], e->slab, err) &&
              dalloc<double2>(e->OUT, e->slab, err) && dalloc<double2>(e->PSI, e->slab, err) &&
              dalloc<double2>(e->PSI0, e->slab, err) && dalloc<double2>(e->TGT, e->slab, err) &&
              dalloc<double2>(e->CHI, e->slab, err) && dalloc<double2>(e->X, e->slab * (size_t)(N_T + 1), err) &&
              dalloc<double>(e->partial, (size_t)L * e->n_partial, err) && dalloc<int>(e->d_col_of_traj, (size_t)N, err) &&
              dalloc<int>(e->d_traj_of_col, (size_t)e->ld, err);
    if (ok && !e->hermitian && !e->sparse) ok = dalloc<double2>(e->Hb, (size_t)n_gen * (1 + L) * mat, err);
    if (ok && store_fw) ok = dalloc<double2>(e->PHI, e->slab * (size_t)(N_T + 1), err);
    // Stream-K for the DMMA GEMM when the row blocks would leave SMs idle (C5: 128 row blocks on 148 SMs) and K is
    // long enough to split: as many CTAs as SMs, each total/G chunks of the (row block, k) space.
    {
        const int R = e->dp / BM, nk = e->dp / BK, G = e->sm_count;
        e->streamk = !e->sparse && R >= 32 && R < G && nk >= 32 && (G + R - 1) / R + 1 <= kSkParts && !getenv("KROTOV_NO_STREAMK");
        if (ok && e->streamk) {
            ok = dalloc<double2>(e->sk_ws, (size_t)R * kSkParts * BM * 64, err) &&
                 dalloc<unsigned>(e->sk_flags, (size_t)R * kSkParts * 4, err);
            if (ok) cudaMemsetAsync(e->sk_flags.get<unsigned>(), 0, (size_t)R * kSkParts * 4 * sizeof(unsigned), e->stream);
        }
    }
    if (ok && e->sparse)
        ok = dalloc<int>(e->ell_cols, nslots, err) && dalloc<double2>(e->Pvf, (size_t)n_gen * (1 + L) * nslots, err) &&
             dalloc<double2>(e->Gv, (size_t)n_gen * nslots, err) &&
             (e->hermitian || dalloc<double2>(e->Pvb, (size_t)n_gen * (1 + L) * nslots, err));
    if (!ok) return nullptr;
    if (e->sparse) {
        // ELL arrays padded to dp rows: padding rows / slots point at their own row with value 0
        std::vector<int> cols(nslots);
        for (size_t i = 0; i < (size_t)e->dp; ++i)
            for (int sl = 0; sl < e->W; ++sl)
                cols[i * e->W + sl] = (i < (size_t)d) ? (*sp->cols)[i * e->W + sl] : (int)i;
        copy_to_device(e->ell_cols.get<int>(), cols.data(), nslots * 4, e->stream, true);
        std::vector<cplx> vbuf(nslots);
        for (int dir = 0; dir < (e->hermitian ? 1 : 2); ++dir) {
            const std::vector<cplx> &src = dir == 0 ? *sp->vals_f : *sp->vals_b;
            double2 *dst = dir == 0 ? e->Pvf.get<double2>() : e->Pvb.get<double2>();
            for (int q = 0; q < n_gen * (1 + L); ++q) {
                std::fill(vbuf.begin(), vbuf.end(), cplx(0, 0));
                memcpy(vbuf.data(), &src[(size_t)q * d * e->W], sizeof(cplx) * (size_t)d * e->W);
                copy_to_device(dst + (size_t)q * nslots, vbuf.data(), nslots * 16, e->stream, true);
            }
        }
    }
    if ((e->sparse && !sweep_configure(e.get())) || (!e->sparse && !dsweep_configure(e.get()))) {
        err = "dense_create: allocation for the persistent sweep failed";
        return nullptr;
    }
    // upload padded generator terms (and adjoints), states, targets
    std::vector<cplx> buf(mat);
    for (int q = 0; !e->sparse && q < n_gen * (1 + L); ++q) {
        const cplx *M = &Hdense[(size_t)q * d * d];
        std::fill(buf.begin(), buf.end(), cplx(0, 0));
        for (int i = 0; i < d; ++i) memcpy(&buf[(size_t)i * e->dp], &M[(size_t)i * d], sizeof(cplx) * d);
        copy_to_device(e->Hf.get<double2>() + (size_t)q * mat, buf.data(), mat * 16, e->stream, true);
        if (!e->hermitian) {
            std::fill(buf.begin(), buf.end(), cplx(0, 0));
            for (int i = 0; i < d; ++i)
                for (int j = 0; j < d; ++j) buf[(size_t)i * e->dp + j] = std::conj(M[(size_t)j * d + i]);
            copy_to_device(e->Hb.get<double2>() + (size_t)q * mat, buf.data(), mat * 16, e->stream, true);
        }
    }
    auto to_block = [&](const double *src, double2 *dst) {
        std::vector<cplx> blk(e->slab, cplx(0, 0));
        if (src) {
            const cplx *s = reinterpret_cast<const cplx *>(src);
            for (int k = 0; k < N; ++k)
                for (int i = 0; i < d; ++i) blk[(size_t)i * e->ld + e->col_of_traj[k]] = s[(size_t)k * d + i];
        }
        copy_to_device(dst, blk.data(), e->slab * 16, e->stream, true);
    };
    to_block(psi0, e->PSI0.get<double2>());
    to_block(target, e->TGT.get<double2>());
    cudaMemsetAsync(e->CHI.get<double2>(), 0, e->slab * 16, e->stream);
    cudaMemsetAsync(e->PSI.get<double2>(), 0, e->slab * 16, e->stream);
    copy_to_device(e->d_col_of_traj.get<int>(), e->col_of_traj.data(), (size_t)N * 4, e->stream, false);
    copy_to_device(e->d_traj_of_col.get<int>(), e->traj_of_col.data(), (size_t)e->ld * 4, e->stream, false);
    if (cudaGetLastError() != cudaSuccess) {
        err = "dense_create: upload failed";
        return nullptr;
    }
    return e.release();
}

void dense_set_comm(DenseEngine *e, const DenseComm &c) { e->comm = c; }

void dense_destroy(DenseEngine *e) { delete e; }

void dense_set_amp(DenseEngine *e, const AmpDev &a) {
    e->amp = a;
    e->cheb_version++;  // the amplitude pointers travel by value in the launch parameters: a captured iteration is stale now
}

void dense_info(DenseEngine *e, krotov_info *out) {
    out->grid_blocks = e->sparse ? (e->sweep_launches ? e->sw_grid : e->dp / SP_ROWS) : (e->streamk ? e->sm_count : e->dp / BM);
    out->graph_replays = e->graph_replays;
    out->block_threads = e->sparse ? SP_WARPS * 32 : GEMM_THREADS;
    if (e->dsweep && e->sweep_launches) {  // the cluster sweep served the last calls
        out->grid_blocks = e->ds_units * kDsCluster;
        out->block_threads = kDsThreads;
    }
    out->kernel = e->kernel_last;
    out->lanes_per_traj = 0;
    out->nnz_union = e->sparse ? e->nnz_union : e->d * e->d;
    out->ell_width = e->sparse ? e->W : 0;
    out->hbm_bytes_state = (int64_t)(e->slab * (size_t)(e->N_T + 1) * 16);
    for (int dir = 0; dir < 2; ++dir) {
        int mm = 0;
        for (int v : e->ch[dir].m) mm = std::max(mm, v);
        (dir == 0 ? out->m_fw : out->m_bw) = mm;
    }
}

bool dense_set_cheby(DenseEngine *e, int direction, int ndtc, const std::vector<int> &dtc_of_step,
                     const std::vector<double> &E_min, const std::vector<double> &Delta, const std::vector<int> &m,
                     const std::vector<double> &coef, int m_max, const std::vector<cplx> &phase, std::string &err) {
    Cheb &c = e->ch[direction];
    const bool same = c.set && c.ndtc == ndtc && c.mmax == m_max && c.dtc_of_step == dtc_of_step && c.E_min == E_min &&
                      c.Delta == Delta && c.m == m && c.coef == coef && c.phase == phase;
    c.ndtc = ndtc; c.mmax = m_max; c.dtc_of_step = dtc_of_step; c.E_min = E_min; c.Delta = Delta; c.m = m;
    c.coef = coef; c.phase = phase; c.set = true;
    if (!same) e->cheb_version++;  // coefficients travel by value in the launch parameters: a captured iteration is stale now
    if ((e->sweep || e->dsweep) && !same) {  // the persistent sweeps read the tables from device memory
        std::vector<double2> ph(phase.size());
        for (size_t i = 0; i < phase.size(); ++i) ph[i] = make_double2(phase[i].real(), phase[i].imag());
        cudaStreamSynchronize(e->stream);
        if (!sweep_upload(e, e->sw_coef[direction], coef, err) || !sweep_upload(e, e->sw_m[direction], m, err) ||
            !sweep_upload(e, e->sw_phase[direction], ph, err) || !sweep_upload(e, e->sw_dtc[direction], dtc_of_step, err) ||
            !sweep_upload(e, e->sw_Emin[direction], E_min, err) || !sweep_upload(e, e->sw_Delta[direction], Delta, err))
            return false;
    }
    for (int v : m)
        if (v < 3) {
            err = "dense path needs at least 3 Chebyshev coefficients per step (Delta * dt too small)";
            return false;
        }
    return true;
}

static bool finish_sweep(DenseEngine *e, double2 *d_tau, std::string &err) {
    tau_kernel<<<(e->N + 3) / 4, 128, 0, e->stream>>>(e->PSI.get<double2>(), e->TGT.get<double2>(), e->d, e->ld,
                                                      e->d_col_of_traj.get<int>(), e->N, d_tau);
    e->launches++;
    DK_CHECK(cudaGetLastError());
    return true;
}

// Psi_k(T) := initial states, tau from them: the state of freshly initialised propagators, which is what the driver
// reads when `skip_initial_forward_propagation` is set (src/optimize.jl:171-181, :297, :378-381)
bool dense_seed(DenseEngine *e, double2 *d_tau, std::string &err) {
    DK_CHECK(cudaMemcpyAsync(e->PSI.get<double2>(), e->PSI0.get<double2>(), e->slab * 16, cudaMemcpyDeviceToDevice, e->stream));
    return finish_sweep(e, d_tau, err);
}

bool dense_forward(DenseEngine *e, const double *d_eps, double2 *d_tau, long long &launches, std::string &err) {
    e->launches = 0;
    e->kernel_last = kernel_kind(e, 0);
    DK_CHECK(cudaMemcpyAsync(e->PSI.get<double2>(), e->PSI0.get<double2>(), e->slab * 16, cudaMemcpyDeviceToDevice, e->stream));
    if (sweep_usable(e, 0)) {
        if (!launch_sweep(e, 0, d_eps, nullptr, nullptr, nullptr, nullptr, err) || !finish_sweep(e, d_tau, err)) return false;
        launches += e->launches;
        return true;
    }
    if (e->store_fw)
        DK_CHECK(cudaMemcpyAsync(e->PHI.get<double2>(), e->PSI0.get<double2>(), e->slab * 16, cudaMemcpyDeviceToDevice, e->stream));
    for (int n = 0; n < e->N_T; ++n)
        if (!step(e, KROTOV_FORWARD, n, gen_coeffs_old(e, d_eps),
                  e->store_fw ? e->PHI.get<double2>() + e->slab * (size_t)(n + 1) : nullptr, err))
            return false;
    if (!finish_sweep(e, d_tau, err)) return false;
    launches += e->launches;
    return true;
}

namespace {
bool iterate_body(DenseEngine *e, const double *d_eps_old, double *d_eps_new, const double *d_alpha,
                  const double *d_dt, double *d_ga, const double2 *d_chi_coef, double2 *d_tau, std::string &err);
}

// One Krotov iteration on the block path.  The iteration is a fixed stream of ~20 launches per time step and
// direction whose parameters do not change between iterations (pulses, chi coefficients, tau live at fixed device
// addresses) until the Chebyshev tables change, so the second time an identical iteration is asked for it is
// captured into ONE CUDA graph and replayed from then on.  Measured (tools/gpu_graph_bench.py): dense d = 100, 20
// trajectories, 3603 launches per iteration: 45.1 -> 36.9 ms; capture + instantiation cost ~9 us per node once, so
// the graph is built only when two consecutive iterations were identical (tables settled) and the iteration has at
// most kGraphMaxNodes launches (C5 has 500 000 and is compute-bound anyway).  Not with several ranks (the mailbox
// parity alternates).
constexpr long long kGraphMaxNodes = 60000;

bool dense_iterate(DenseEngine *e, const double *d_eps_old, double *d_eps_new, const double *d_alpha,
                   const double *d_dt, double *d_ga, const double2 *d_chi_coef, double2 *d_tau, long long &launches,
                   std::string &err) {
    DenseEngine::GraphKey key;
    key.cheb_version = e->cheb_version;
    e->kernel_last = kernel_kind(e, 1);
    const void *ptrs[8] = {d_eps_old, d_eps_new, d_alpha, d_dt, d_ga, d_chi_coef, d_tau, e->amp.amp_old};
    memcpy(key.ptr, ptrs, sizeof(ptrs));
    const bool graph_ok = e->comm.world <= 1 && !getenv("KROTOV_NO_GRAPH") && !sweep_usable(e, 1);  // (the sweep is 3 launches)
    if (graph_ok && e->graph_exec != nullptr && e->graph_key == key) {
        DK_CHECK(cudaGraphLaunch(e->graph_exec, e->stream));
        launches += e->graph_launches;
        e->graph_replays++;
        e->chi_from_host = false;
        return true;
    }
    if (e->graph_exec != nullptr) {
        cudaGraphExecDestroy(e->graph_exec);
        e->graph_exec = nullptr;
    }
    const bool capture = graph_ok && e->last_key == key && e->stable_iterations >= 2 && e->last_launches > 0 &&
                         e->last_launches <= kGraphMaxNodes;
    if (capture) DK_CHECK(cudaStreamBeginCapture(e->stream, cudaStreamCaptureModeThreadLocal));
    e->launches = 0;
    const bool ok = iterate_body(e, d_eps_old, d_eps_new, d_alpha, d_dt, d_ga, d_chi_coef, d_tau, err);
    if (capture) {
        cudaGraph_t graph = nullptr;
        const cudaError_t ce = cudaStreamEndCapture(e->stream, &graph);
        if (!ok) {
            if (graph) cudaGraphDestroy(graph);
            return false;
        }
        if (ce != cudaSuccess || graph == nullptr) {
            err = std::string("cudaStreamEndCapture: ") + cudaGetErrorString(ce);
            return false;
        }
        const cudaError_t ci = cudaGraphInstantiate(&e->graph_exec, graph, 0);
        cudaGraphDestroy(graph);
        if (ci != cudaSuccess) {
            e->graph_exec = nullptr;
            err = std::string("cudaGraphInstantiate: ") + cudaGetErrorString(ci);
            return false;
        }
        e->graph_key = key;
        e->graph_launches = e->launches;
        DK_CHECK(cudaGraphLaunch(e->graph_exec, e->stream));
    } else if (!ok) {
        return false;
    }
    e->stable_iterations = (e->last_key == key) ? e->stable_iterations + 1 : 1;
    e->last_key = key;
    e->last_launches = e->launches;
    e->chi_from_host = false;
    launches += e->launches;
    return true;
}

namespace {
bool iterate_body(DenseEngine *e, const double *d_eps_old, double *d_eps_new, const double *d_alpha,
                  const double *d_dt, double *d_ga, const double2 *d_chi_coef, double2 *d_tau, std::string &err) {
    const int N_T = e->N_T;
    // ---- chi(T)
    if (d_chi_coef != nullptr) {
        chi_from_coef_kernel<<<e->sm_count * 2, 256, 0, e->stream>>>(e->CHI.get<double2>(), e->TGT.get<double2>(), d_chi_coef,
                                                                     e->d_traj_of_col.get<int>(),
                                                                     e->dp, e->ld);
        e->launches++;
    }
    if (sweep_usable(e, 1))
        return launch_sweep(e, 1, d_eps_old, d_eps_new, d_alpha, d_dt, d_ga, err) && finish_sweep(e, d_tau, err);
    // ---- backward sweep: chi(t_n) for all n into X
    DK_CHECK(cudaMemcpyAsync(e->PSI.get<double2>(), e->CHI.get<double2>(), e->slab * 16, cudaMemcpyDeviceToDevice, e->stream));
    DK_CHECK(cudaMemcpyAsync(e->X.get<double2>() + e->slab * (size_t)N_T, e->CHI.get<double2>(), e->slab * 16,
                             cudaMemcpyDeviceToDevice, e->stream));
    for (int n = N_T - 1; n >= 0; --n)
        if (!step(e, KROTOV_BACKWARD, n, gen_coeffs_old(e, d_eps_old), e->X.get<double2>() + e->slab * (size_t)n, err)) return false;
    // ---- forward sweep with sequential update
    DK_CHECK(cudaMemcpyAsync(e->PSI.get<double2>(), e->PSI0.get<double2>(), e->slab * 16, cudaMemcpyDeviceToDevice, e->stream));
    const size_t mat = (size_t)e->dp * e->dp;
    const int ctas = e->dp / BM;
    for (int n = 0; n < N_T; ++n) {
        for (int l = 0; l < e->L; ++l) {
            for (size_t bi = 0; bi < e->blocks.size(); ++bi) {
                const Block &b = e->blocks[bi];
                GemmParams p;
                memset(&p, 0, sizeof(p));
                p.A = e->Hf.get<double2>() + ((size_t)b.g * (1 + e->L) + 1 + l) * mat;  // mu_l = H_l (src/optimize.jl:275-276)
                p.B = e->PSI.get<double2>();
                p.epi = 1;
                p.CHI = e->X.get<double2>() + e->slab * (size_t)n;
                if (e->sparse) {
                    p.partial = e->partial.get<double>() + (size_t)l * e->n_partial;
                    const double2 *mu = e->Pvf.get<double2>() + ((size_t)b.g * (1 + e->L) + 1 + l) * ((size_t)e->dp * e->W);
                    if (!launch_spmm(e, b, mu, p, e->sp_part_off[bi], err)) return false;
                    continue;
                }
                p.partial = e->partial.get<double>() + (size_t)l * e->n_partial + bi * ctas;
                if (!launch_gemm(e, b, p, err)) return false;
            }
        }
        if (e->amp.tie != nullptr)
            update_tied_kernel<<<1, 32, 0, e->stream>>>(e->partial.get<double>(), e->n_partial, e->L, d_alpha, d_eps_old, d_eps_new,
                                                        d_ga, d_dt, N_T, n, e->comm, e->amp);
        else
            update_kernel<<<e->L, 32, 0, e->stream>>>(e->partial.get<double>(), e->n_partial, e->L, d_alpha, d_eps_old, d_eps_new, d_ga,
                                                     d_dt, N_T, n, e->comm, e->amp);
        e->launches++;
        if (!step(e, KROTOV_FORWARD, n, gen_coeffs_new(e, d_eps_new),
                  e->store_fw ? e->PHI.get<double2>() + e->slab * (size_t)n : nullptr, err))
            return false;
    }
    return finish_sweep(e, d_tau, err);
}
}  // namespace

bool dense_set_chi(DenseEngine *e, const double *chi_host, std::string &err) {
    std::vector<cplx> blk(e->slab, cplx(0, 0));
    const cplx *s = reinterpret_cast<const cplx *>(chi_host);
    for (int k = 0; k < e->N; ++k)
        for (int i = 0; i < e->d; ++i) blk[(size_t)i * e->ld + e->col_of_traj[k]] = s[(size_t)k * e->d + i];
    DK_CHECK(copy_to_device(e->CHI.get<double2>(), blk.data(), e->slab * 16, e->stream, true));
    e->chi_from_host = true;
    return true;
}

bool dense_get_states(DenseEngine *e, double *states_host, std::string &err) {
    std::vector<cplx> blk(e->slab);
    DK_CHECK(cudaMemcpy(blk.data(), e->PSI.get<double2>(), e->slab * 16, cudaMemcpyDeviceToHost));
    cplx *o = reinterpret_cast<cplx *>(states_host);
    for (int k = 0; k < e->N; ++k)
        for (int i = 0; i < e->d; ++i) o[(size_t)k * e->d + i] = blk[(size_t)i * e->ld + e->col_of_traj[k]];
    return true;
}

bool dense_get_storage(DenseEngine *e, int which, int k, int n0, int n1, double *out_host, std::string &err) {
    const double2 *S = which == KROTOV_FORWARD ? e->PHI.get<double2>() : e->X.get<double2>();
    const int c = e->col_of_traj[k];
    cplx *o = reinterpret_cast<cplx *>(out_host);
    std::vector<cplx> colbuf(e->d);
    for (int n = n0; n < n1; ++n) {
        // column c of slot n: strided gather (one 2-D copy per slot)
        DK_CHECK(cudaMemcpy2D(colbuf.data(), 16, S + e->slab * (size_t)n + c, (size_t)e->ld * 16, 16, e->d,
                              cudaMemcpyDeviceToHost));
        memcpy(o + (size_t)(n - n0) * e->d, colbuf.data(), (size_t)e->d * 16);
    }
    return true;
}

}  // namespace kr
