// Persistent sweep for MODERATE dense generators (32 < d <= kDsMaxD): the whole Krotov iteration in one cooperative
// launch of thread-block clusters, no kernel boundary between Chebyshev terms or time steps.
//
// The launch-per-term stream of the DMMA path (dense_gemm_kernel + build_G_kernel + update_kernel, ~20 launches per
// time step) costs 5-16 us per term on generators whose term is 0.1-1 us of arithmetic.  Here a CLUSTER of 8 CTAs owns
// a group of <= 8 trajectories (columns of the state block) of one generator:
//   * CTA r of the cluster owns rows [r R, (r+1) R) of the generator, R = ceil(d / 8); its slice of
//     G = 2c (H_0 - beta + sum_l a_l H_l) is rebuilt in SHARED memory once per time step from the term slices in L2;
//   * every CTA holds the full V_{j-1} of its column group in shared memory (8 x d complex, transposed); warp w forms
//     the 8 rows x 8 columns tile w of V_j = G V_{j-1} + V_{j-2} on the FP64 tensor pipe: per 4 values of k one
//     16-byte fragment load of G and one of V feed four `mma.sync.m8n8k4.f64` (DMMA: Gr Vr, -Gi Vi, Gr Vi, Gi Vr).
//     (A first version formed one element per thread with DFMA: two 16-byte shared-memory loads per 4 FMA made it
//     crossbar-bound at 45 / 95 us per step and direction for d = 100 / 200 -- the fragment form moves 1/8 of that.)
//     V_{j-2}, the running sum and the own elements stay in registers;
//   * the new rows go to a ping-pong exchange block in L2, ONE cluster barrier (barrier.cluster, ~380 cycles) orders
//     them, and every CTA of the cluster reloads the full column group -- the column groups never talk to each other
//     inside a time step;
//   * once per time step of the forward sweep the overlap sums Im<chi|H_l|psi> of all clusters meet: CTA partials,
//     one grid barrier (the counter barrier of the sparse sweep), every CTA adds them in the same fixed order.
// Same state blocks, storage slots, Chebyshev tables and per-element arithmetic as the launch stream
// (build_G_kernel / dense_gemm_kernel epilogues / update_kernel): tested against it.
// Reference: the time loop of src/optimize.jl:303-317 (backward) and :328-370 (update + forward).
#pragma once

namespace kr {
namespace {

constexpr int kDsCluster = 8;    // CTAs per cluster = row slices of the generator
constexpr int kDsCols = 8;       // trajectories (columns) per cluster
constexpr int kDsThreads = 256;
constexpr int kDsMaxD = 256;     // 8 warps x 8 rows per CTA = 64 rows per slice; slice + column group must fit 227 KB
// shared-memory row stride (in 16-byte words) for k-extent d: >= d rounded up to 4, and = 4 (mod 8) so that the 8 lanes
// of a quarter-warp (2 rows x 4 consecutive k) of a fragment load hit 8 different 16-byte bank groups
__host__ __device__ constexpr int ds_stride(int d) { return ((d + 3) / 4 * 4 + 7) / 8 * 8 + 4; }

struct DSweepParams {
    int d, dp, ld, L, N_T, mode, store_fw;
    int n_units;               // clusters that carry work; unit u = (generator, first column, columns)
    int R;                     // rows per CTA
    int gpad;                  // row stride of the generator slice and of the transposed column group in shared memory
    const int *units;          // [n_units][3]
    const double2 *H[2];       // per direction: [g][1+L][dp][dp] row-major dense terms
    const double *coef[2];
    const int *m[2];
    const double2 *phase[2];
    const int *dtc[2];
    const double *E_min[2], *Delta[2];
    int ndtc[2], mmax[2];
    double2 *PSI, *X, *PHI, *VX[2];
    const double2 *PSI0, *CHI;
    size_t slab;
    const double *eps_old, *alpha, *dt, *amp_old;
    double *eps_new, *ga;
    double *partial;           // [L][gridDim.x]
    unsigned *bar;
    AmpDev am;
    DenseComm cm;              // several ranks: mailboxes of this iteration's parity
    long long *prof;           // optional [8] cycle counters of CTA 0 (KROTOV_PROF=1): build G, tiles, exchange store +
                               // cluster barrier, group reload, overlaps, grid barrier + update
};

__device__ __forceinline__ unsigned ds_cluster_rank() {
    unsigned r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void ds_cluster_sync() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

__device__ __forceinline__ void ds_grid_barrier(unsigned *bar, unsigned &target) {
    __syncthreads();
    if (threadIdx.x == 0) {
        target += gridDim.x;
        __threadfence();
        asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(bar) : "memory");
        while ((int)(ld_acquire_u32(bar) - target) < 0) {
        }
        __threadfence();
    }
    __syncthreads();
}

// C(8 x 8 tile) = A(8 rows of the slice) . V(column group) over k in [k0, k1), complex, on the FP64 tensor pipe.
// `ga` -> this lane's row of the A fragment (row gid of the tile, k offset tig), `vb` -> this lane's column of the
// transposed group (column gid, k offset tig).  On return the lane holds C[gid][2 tig] = (cr0, ci0) and
// C[gid][2 tig + 1] = (cr1, ci1).  Four independent accumulator pairs: back-to-back DMMAs into one pair wait for each
// other (measured 88 cycles per k-step of 4 DMMAs against 64 of issue).
__device__ __forceinline__ void ds_tile(const double2 *__restrict__ ga, const double2 *__restrict__ vb, const int k0,
                                        const int k1, double &cr0, double &cr1, double &ci0, double &ci1) {
    double pr0 = 0.0, pr1 = 0.0, qr0 = 0.0, qr1 = 0.0, pi0 = 0.0, pi1 = 0.0, qi0 = 0.0, qi1 = 0.0;
#pragma unroll 4
    for (int k = k0; k < k1; k += 4) {
        const double2 a = ga[k], b = vb[k];
        dmma(pr0, pr1, a.x, b.x);
        dmma(pi0, pi1, a.x, b.y);
        dmma(qr0, qr1, -a.y, b.y);
        dmma(qi0, qi1, a.y, b.x);
    }
    cr0 = pr0 + qr0;
    cr1 = pr1 + qr1;
    ci0 = pi0 + qi0;
    ci1 = pi1 + qi1;
}

// shared memory (transposed, [column][k], zero padded) <- the column group of a state block in global memory.  All loads
// of a thread are in flight before the first store (a dependent loop cost 1.4 us per Chebyshev term at d = 200).
__device__ __forceinline__ void ds_load_group(double2 *vt, const double2 *src, const int d, const int d4, const int vpad,
                                              const int ld, const int col0, const int ncols) {
    constexpr int U = 4;
    const int total = d4 * kDsCols;
    for (int base = threadIdx.x; base < total; base += U * kDsThreads) {
        double2 v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int i = base + u * kDsThreads;
            const int k = i / kDsCols, c = i - k * kDsCols;
            v[u] = (i < total && c < ncols && k < d) ? __ldcg(src + (size_t)k * ld + col0 + c) : make_double2(0.0, 0.0);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int i = base + u * kDsThreads;
            const int k = i / kDsCols, c = i - k * kDsCols;
            if (i < total) vt[(size_t)c * vpad + k] = v[u];
        }
    }
    __syncthreads();
}

__global__ void __launch_bounds__(kDsThreads, 1) dense_cluster_sweep_kernel(const __grid_constant__ DSweepParams p) {
    extern __shared__ __align__(16) unsigned char ds_smem[];
    __shared__ double wsum[kMaxL][kDsThreads / 32];
    __shared__ double eps_sh[kMaxL];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int crank = (int)ds_cluster_rank();
    const int unit = blockIdx.x / kDsCluster;
    const bool live = unit < p.n_units;
    const int g = live ? p.units[unit * 3] : 0, col0 = live ? p.units[unit * 3 + 1] : 0, ncols = live ? p.units[unit * 3 + 2] : 0;
    const int d = p.d, R = p.R, gpad = p.gpad, d4 = (d + 3) / 4 * 4, R8 = (R + 7) / 8 * 8;
    const int row0 = crank * R, nrows = max(0, min(R, d - row0));
    double2 *gs = reinterpret_cast<double2 *>(ds_smem);  // [R8][gpad] generator slice (also stages the H_l slices)
    double2 *vs = gs + (size_t)R8 * gpad;                // [8][gpad] V_{j-1} of the column group, transposed
    const size_t mat = (size_t)p.dp * p.dp;
    // warp w owns the 8 x 8 output tile of slice rows [8 w, 8 w + 8); DMMA accumulator layout: lane (gid, tig) holds
    // row gid, columns 2 tig and 2 tig + 1
    // With few tiles (R <= 32: 4 tiles or fewer) the k range of a tile is split over two warps, whose partial tiles
    // meet in shared memory: all 8 warps (all four tensor pipes twice) work on every term.
    constexpr int kDsMaxOut = 2;
    constexpr int kWarps = kDsThreads / 32;
    const int gid = lane >> 2, tig = lane & 3;
    const int ntiles = R8 / 8;
    const bool split = 2 * ntiles <= kWarps;
    const int tile = split ? warp % ntiles : warp, khalf = split ? warp / ntiles : 0;
    const bool tile_live = live && tile * 8 < nrows && (split ? khalf < 2 : true);
    const int kmid = split ? (d4 / 8) * 4 : d4;  // multiple of 4
    const int k_lo = khalf == 0 ? 0 : kmid, k_hi = (split && khalf == 0) ? kmid : d4;
    const bool owner = tile_live && khalf == 0;  // the warp that finishes the tile (epilogue, stores)
    int orow[kDsMaxOut], ocol[kDsMaxOut];
    bool oval[kDsMaxOut];
#pragma unroll
    for (int q = 0; q < kDsMaxOut; ++q) {
        orow[q] = tile * 8 + gid;
        ocol[q] = 2 * tig + q;
        oval[q] = owner && orow[q] < nrows && ocol[q] < ncols;
    }
    const double2 *ga = gs + (size_t)(tile * 8 + gid) * gpad + tig;  // A fragment: row gid of the tile, k offset tig
    const double2 *vb = vs + (size_t)gid * gpad + tig;               // B fragment: column gid, k offset tig
    __shared__ double part_sm[kWarps / 2][32][4];                    // partial tiles of the second k half
    // tile product of this warp's share; after it the owner lanes hold the complete (tr, ti)
    auto tile_product = [&](double (&tr)[kDsMaxOut], double (&ti)[kDsMaxOut]) {
        tr[0] = tr[1] = ti[0] = ti[1] = 0.0;
        if (tile_live) ds_tile(ga, vb, k_lo, k_hi, tr[0], tr[1], ti[0], ti[1]);  // warp-uniform: mma.sync needs the whole warp
        if (split) {
            if (tile_live && khalf == 1) {
                part_sm[tile][lane][0] = tr[0];
                part_sm[tile][lane][1] = tr[1];
                part_sm[tile][lane][2] = ti[0];
                part_sm[tile][lane][3] = ti[1];
            }
            __syncthreads();
            if (owner) {
                tr[0] += part_sm[tile][lane][0];
                tr[1] += part_sm[tile][lane][1];
                ti[0] += part_sm[tile][lane][2];
                ti[1] += part_sm[tile][lane][3];
            }
        }
    };
    unsigned bar_target = 0;
    long long pc[6] = {0, 0, 0, 0, 0, 0};
    const bool prof = p.prof != nullptr && blockIdx.x == 0 && tid == 0;
#define DS_T(i, stmt)                          \
    do {                                       \
        const long long t_ = clock64();        \
        stmt;                                  \
        if (prof) pc[i] += clock64() - t_;     \
    } while (0)

    // generator slice for interval n of direction dir with coefficients cf[]  (build_G_kernel's arithmetic)
    auto build_G = [&](const int dir, const double (&cf)[kMaxL]) {
        const double sc = 4.0 / p.Delta[dir][g], beta = p.Delta[dir][g] / 2 + p.E_min[dir][g];
        const double2 f = (dir == KROTOV_FORWARD) ? make_double2(0.0, -sc) : make_double2(0.0, sc);
        const double2 *H = p.H[dir] + (size_t)g * (1 + p.L) * mat;
        constexpr int U = 4;  // U elements per thread with all their loads in flight (L2 latency, not bandwidth, bound this)
        const int total = R8 * d4;
        for (int base = tid; base < total; base += U * kDsThreads) {
            double2 h[U];
            bool ok[U];
            size_t src[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int i = base + u * kDsThreads, r = i / d4, k = i - r * d4;
                ok[u] = i < total && r < nrows && k < d;
                src[u] = ok[u] ? (size_t)(row0 + r) * p.dp + k : 0;
                h[u] = ok[u] ? H[src[u]] : make_double2(0.0, 0.0);
                if (ok[u] && row0 + r == k) h[u].x -= beta;
            }
            for (int l = 0; l < p.L; ++l) {
                double2 hl[U];
#pragma unroll
                for (int u = 0; u < U; ++u) hl[u] = ok[u] ? H[(size_t)(l + 1) * mat + src[u]] : make_double2(0.0, 0.0);
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    h[u].x = fma(cf[l], hl[u].x, h[u].x);
                    h[u].y = fma(cf[l], hl[u].y, h[u].y);
                }
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int i = base + u * kDsThreads, r = i / d4, k = i - r * d4;
                // rows / columns beyond the slice: zero padding of the fragments
                if (i < total) gs[(size_t)r * gpad + k] = ok[u] ? make_double2(f.x * h[u].x - f.y * h[u].y, f.x * h[u].y + f.y * h[u].x)
                                                                 : make_double2(0.0, 0.0);
            }
        }
        __syncthreads();
    };

    // one propagation step of the cluster's column group: PSI <- exp(-/+ i H dt) PSI, result also into `store`
    auto step = [&](const int dir, const int n, double2 *store) {
        const int ci = g * p.ndtc[dir] + p.dtc[dir][n];
        const int m = live ? p.m[dir][ci] : 0;
        const double2 ph = p.phase[dir][ci];
        const double *a = p.coef[dir] + (size_t)ci * p.mmax[dir];
        const double a0 = a[0];
        double2 vm1[kDsMaxOut], vm2[kDsMaxOut], out[kDsMaxOut];
        if (live) ds_load_group(vs, p.PSI, d, d4, gpad, p.ld, col0, ncols);
#pragma unroll
        for (int q = 0; q < kDsMaxOut; ++q) {
            vm1[q] = oval[q] ? vs[(size_t)ocol[q] * gpad + row0 + orow[q]] : make_double2(0.0, 0.0);
            vm2[q] = make_double2(0.0, 0.0);
            out[q] = make_double2(a0 * vm1[q].x, a0 * vm1[q].y);
        }
        for (int j = 1; j < m; ++j) {
            const double aj = a[j];
            const bool last = (j == m - 1);
            double2 *vx = p.VX[j & 1];
            double tr[kDsMaxOut] = {0.0, 0.0}, ti[kDsMaxOut] = {0.0, 0.0};
            const long long t_tile = clock64();
            tile_product(tr, ti);
            if (prof) pc[1] += clock64() - t_tile;
            const long long t_x = clock64();
#pragma unroll
            for (int q = 0; q < kDsMaxOut; ++q) {
                if (!oval[q]) continue;
                const double cr = tr[q], ci_ = ti[q];
                double2 v;
                if (j == 1)
                    v = make_double2(0.5 * cr, 0.5 * ci_);
                else
                    v = make_double2(cr + vm2[q].x, ci_ + vm2[q].y);
                out[q] = make_double2(fma(aj, v.x, out[q].x), fma(aj, v.y, out[q].y));
                vm2[q] = vm1[q];
                vm1[q] = v;
                const size_t idx = (size_t)(row0 + orow[q]) * p.ld + col0 + ocol[q];
                if (last) {
                    const double2 r = make_double2(ph.x * out[q].x - ph.y * out[q].y, ph.x * out[q].y + ph.y * out[q].x);
                    p.PSI[idx] = r;
                    if (store) store[idx] = r;
                } else {
                    vx[idx] = v;
                }
            }
            if (!last) {
                ds_cluster_sync();  // every row slice of V_j is in L2
                if (prof) pc[2] += clock64() - t_x;
                DS_T(3, ds_load_group(vs, vx, d, d4, gpad, p.ld, col0, ncols));
            }
        }
        DS_T(2, ds_cluster_sync());  // PSI of the column group is complete (the next step, or the overlaps, read all rows)
    };

    const size_t gtid = (size_t)blockIdx.x * blockDim.x + tid, gthreads = (size_t)gridDim.x * blockDim.x;
    double cf[kMaxL];
#pragma unroll
    for (int l = 0; l < kMaxL; ++l) cf[l] = 0.0;

    if (p.mode == 1) {
        // ---- backward sweep: chi(t_n) for all n into X  (src/optimize.jl:303-317)
        for (size_t i = gtid; i < p.slab; i += gthreads) {
            const double2 v = p.CHI[i];
            p.PSI[i] = v;
            p.X[p.slab * (size_t)p.N_T + i] = v;
        }
        ds_grid_barrier(p.bar, bar_target);
        for (int n = p.N_T - 1; n >= 0; --n) {
            for (int l = 0; l < p.L; ++l) cf[l] = p.amp_old[(size_t)l * p.N_T + n];
            if (live) DS_T(0, build_G(KROTOV_BACKWARD, cf));
            step(KROTOV_BACKWARD, n, p.X + p.slab * (size_t)n);
        }
        ds_grid_barrier(p.bar, bar_target);
    }
    // ---- forward sweep
    for (size_t i = gtid; i < p.slab; i += gthreads) {
        const double2 v = p.PSI0[i];
        p.PSI[i] = v;
        if (p.store_fw && p.mode == 0) p.PHI[i] = v;
    }
    ds_grid_barrier(p.bar, bar_target);
    for (int n = 0; n < p.N_T; ++n) {
        if (p.mode == 1) {
            // overlaps Im <chi_k(t_n)| mu_l |psi_k(t_n)> of this CTA's rows and columns  (:339-349)
            const long long t_ov = clock64();
            const double2 *CHI = p.X + p.slab * (size_t)n;
            if (live) ds_load_group(vs, p.PSI, d, d4, gpad, p.ld, col0, ncols);
            for (int l = 0; l < p.L; ++l) {
                double acc = 0.0;
                if (live) {
                    const double2 *Hl = p.H[0] + ((size_t)g * (1 + p.L) + 1 + l) * mat;
                    {   // stage the slice of H_l where G will be rebuilt (loads of a thread in flight together)
                        constexpr int U = 4;
                        const int total = R8 * d4;
                        for (int base = tid; base < total; base += U * kDsThreads) {
                            double2 v[U];
#pragma unroll
                            for (int u = 0; u < U; ++u) {
                                const int i = base + u * kDsThreads, r = i / d4, k = i - r * d4;
                                v[u] = (i < total && r < nrows && k < d) ? Hl[(size_t)(row0 + r) * p.dp + k] : make_double2(0.0, 0.0);
                            }
#pragma unroll
                            for (int u = 0; u < U; ++u) {
                                const int i = base + u * kDsThreads, r = i / d4, k = i - r * d4;
                                if (i < total) gs[(size_t)r * gpad + k] = v[u];
                            }
                        }
                    }
                    __syncthreads();
                    double tr[kDsMaxOut], ti[kDsMaxOut];
                    tile_product(tr, ti);
#pragma unroll
                    for (int q = 0; q < kDsMaxOut; ++q) {
                        if (!oval[q]) continue;
                        const double2 ch = CHI[(size_t)(row0 + orow[q]) * p.ld + col0 + ocol[q]];
                        acc += ch.x * ti[q] - ch.y * tr[q];
                    }
                    __syncthreads();
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
                if (lane == 0) wsum[l][warp] = acc;
            }
            __syncthreads();
            if (tid < p.L) {
                double t = 0.0;
                for (int w = 0; w < kDsThreads / 32; ++w) t += wsum[tid][w];
                p.partial[(size_t)tid * gridDim.x + blockIdx.x] = t;
            }
            if (prof) pc[4] += clock64() - t_ov;
            const long long t_gb = clock64();
            ds_grid_barrier(p.bar, bar_target);
            // every CTA adds the CTA partials in the same fixed order: the same bits everywhere, no broadcast
            if (warp == 0) {
                for (int l = 0; l < p.L; ++l) {
                    double sacc = 0.0;
                    for (int c = lane; c < (int)gridDim.x; c += 32) sacc += __ldcg(p.partial + (size_t)l * gridDim.x + c);
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) sacc += __shfl_xor_sync(0xffffffffu, sacc, o);
                    if (lane == 0) {
                        const double al = p.alpha[(size_t)l * p.N_T + n];
                        sacc = rank_sum_lane(p.cm, p.L, n, l, sacc, blockIdx.x == 0);
                        if (p.am.tie != nullptr) {
                            eps_sh[l] = sacc;  // tied control terms: the update waits for the sums of all terms
                        } else {
                            if (p.am.dfac != nullptr) sacc = __dmul_rn(p.am.dfac[(size_t)l * p.N_T + n], sacc);
                            const double e_new = __dadd_rn(p.eps_old[(size_t)l * p.N_T + n], __dmul_rn(al, sacc));  // :355-356
                            eps_sh[l] = amp_apply(p.am, l, p.N_T, n, e_new);
                            if (blockIdx.x == 0) {
                                p.eps_new[(size_t)l * p.N_T + n] = e_new;
                                const double prev = (n == 0) ? 0.0 : p.ga[l];
                                p.ga[l] = __dadd_rn(prev, __dmul_rn(__dmul_rn(al, __dmul_rn(fabs(sacc), fabs(sacc))), p.dt[n]));  // :357
                            }
                        }
                    }
                }
                if (p.am.tie != nullptr && lane == 0)
                    tie_update_cold(&p, n, eps_sh, blockIdx.x == 0);
            }
            __syncthreads();
            for (int l = 0; l < p.L; ++l) cf[l] = eps_sh[l];
            __syncthreads();
            if (prof) pc[5] += clock64() - t_gb;
        } else {
            for (int l = 0; l < p.L; ++l) cf[l] = p.amp_old[(size_t)l * p.N_T + n];
        }
        double2 *store = nullptr;
        if (p.store_fw) store = p.PHI + p.slab * (size_t)(p.mode == 1 ? n : n + 1);  // slot n in an iteration (sic, :367)
        if (live) DS_T(0, build_G(KROTOV_FORWARD, cf));
        step(KROTOV_FORWARD, n, store);
    }
    if (prof)
        for (int i = 0; i < 6; ++i) p.prof[i] = pc[i];
#undef DS_T
}

}  // namespace
}  // namespace kr
