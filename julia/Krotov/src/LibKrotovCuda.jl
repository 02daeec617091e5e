# ccall bindings for libkrotov_cuda (include/krotov_cuda.h), one Julia function per C entry point.
#
# NOT EXECUTED IN THIS REPOSITORY: Julia is not installed in the build image.  tests/test_host.py parses this file and
# compares the `Problem` / `Info` field lists and every `ccall` signature with the header.
module LibKrotovCuda

const lib = get(ENV, "LIBKROTOV_CUDA", "libkrotov_cuda")

const KROTOV_ABI_VERSION = Cint(1)
const KROTOV_GEN_DENSE_COLMAJOR, KROTOV_GEN_CSR = Cint(0), Cint(1)
const KROTOV_FORWARD, KROTOV_BACKWARD = Cint(0), Cint(1)
const KROTOV_CHI_HOST, KROTOV_CHI_SM, KROTOV_CHI_SS, KROTOV_CHI_RE = Cint(0), Cint(1), Cint(2), Cint(3)
const KROTOV_PATH_WARP, KROTOV_PATH_DENSE, KROTOV_PATH_SPARSE = Cint(1), Cint(2), Cint(3)
const KROTOV_KERNEL_TINY, KROTOV_KERNEL_PREG, KROTOV_KERNEL_SEQ_PREG, KROTOV_KERNEL_PAIR, KROTOV_KERNEL_RELOAD = Cint(1), Cint(2), Cint(3), Cint(4), Cint(5)
const KROTOV_KERNEL_DMMA_STREAM, KROTOV_KERNEL_DENSE_SWEEP, KROTOV_KERNEL_SPARSE_SWEEP, KROTOV_KERNEL_SPARSE_STREAM = Cint(6), Cint(7), Cint(8), Cint(9)
const KROTOV_KERNEL_TAYLOR = Cint(10)
const KROTOV_PROP_CHEBY, KROTOV_PROP_EXPMV = Cint(0), Cint(1)
const COMM_DESC_BYTES = 256

# mirrors `krotov_problem` field by field
struct Problem
    struct_size::Int32
    d::Int32
    n_traj::Int32
    n_ctrl::Int32
    n_steps::Int32
    n_gen::Int32
    gen_format::Int32
    nnz::Int32
    tlist::Ptr{Float64}
    gen_of_traj::Ptr{Int32}
    csr_rowptr::Ptr{Int32}
    csr_colind::Ptr{Int32}
    gen_values::Ptr{Float64}
    term_present::Ptr{UInt8}
    psi0::Ptr{Float64}
    target::Ptr{Float64}
    weight::Ptr{Float64}
    update_shape::Ptr{Float64}
    lambda_a::Ptr{Float64}
    functional::Int32
    n_traj_global::Int32
    store_fw::Int32
    device::Int32
    force_path::Int32
    replicated_forward::Int32
    propagator::Int32
    reserved::NTuple{5,Int32}
end

# mirrors `krotov_info` field by field
struct Info
    struct_size::Int32
    path::Int32
    ell_width::Int32
    nnz_union::Int32
    grid_blocks::Int32
    block_threads::Int32
    m_fw::Int32
    m_bw::Int32
    sm_count::Int32
    exchange::Int32
    launches_total::Int64
    launches_last::Int64
    ms_last::Float64
    ms_last_backward::Float64
    hbm_bytes_state::Int64
    fallback_steps::Int64
    graph_replays::Int64
    ms_rank_wait::Float64
    kernel::Int32
    lanes_per_traj::Int32
    reserved::NTuple{2,Int64}
end

mutable struct Handle
    ptr::Ptr{Cvoid}
    function Handle(ptr)
        h = new(ptr)
        finalizer(destroy, h)
    end
end

function destroy(h::Handle)
    if h.ptr != C_NULL
        ccall((:krotov_destroy, lib), Cint, (Ptr{Cvoid},), h.ptr)
        h.ptr = C_NULL
    end
    nothing
end

abi_version() = ccall((:krotov_abi_version, lib), Cint, ())

last_error(h) = unsafe_string(ccall((:krotov_last_error, lib), Cstring, (Ptr{Cvoid},), h === nothing ? C_NULL : h.ptr))

# a non-zero status becomes an ErrorException carrying the library's text; inside `optimize_krotov` it is caught by the
# try block and recorded as `result.message = "Exception: ..."` unless `rethrow_exceptions=true`
check(h, rc) = rc == 0 ? nothing : error("libkrotov_cuda: " * last_error(h))

function create(p::Problem)
    out = Ref{Ptr{Cvoid}}(C_NULL)
    rc = ccall((:krotov_create, lib), Cint, (Ref{Problem}, Ref{Ptr{Cvoid}}), p, out)
    rc == 0 || error("libkrotov_cuda: " * last_error(nothing))
    Handle(out[])
end

function get_info(h)
    out = Ref{Info}()
    check(h, ccall((:krotov_get_info, lib), Cint, (Ptr{Cvoid}, Ref{Info}), h.ptr, out))
    out[]
end

# m: [n_dt_class, n_gen], coeffs: [m_max, n_dt_class, n_gen] (column-major == [n_gen][n_dt_class][m_max] on the wire)
set_cheby(h, dir, dtc_of_step::Vector{Int32}, dt_of_class::Vector{Float64}, E_min::Vector{Float64},
          Delta::Vector{Float64}, m::Matrix{Int32}, coeffs::Array{Float64,3}) =
    check(h, ccall((:krotov_set_cheby, lib), Cint,
        (Ptr{Cvoid}, Cint, Cint, Ptr{Int32}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Ptr{Float64}, Cint),
        h.ptr, dir, length(dt_of_class), dtc_of_step, dt_of_class, E_min, Delta, m, coeffs, size(coeffs, 1)))

# Taylor settings of a KROTOV_PROP_EXPMV handle: mu, scale: [n_gen]; s, m: [n_dt_class, n_gen];
# coeffs: [m_max, n_dt_class, n_gen] (column-major == [n_gen][n_dt_class][m_max] on the wire)
set_taylor(h, dir, dtc_of_step::Vector{Int32}, dt_of_class::Vector{Float64}, mu::Vector{Float64},
           scale::Vector{Float64}, s::Matrix{Int32}, m::Matrix{Int32}, coeffs::Array{Float64,3}) =
    check(h, ccall((:krotov_set_taylor, lib), Cint,
        (Ptr{Cvoid}, Cint, Cint, Ptr{Int32}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Ptr{Int32}, Ptr{Float64}, Cint),
        h.ptr, dir, length(dt_of_class), dtc_of_step, dt_of_class, mu, scale, s, m, coeffs, size(coeffs, 1)))

# non-linear amplitudes a_l(eps, n) = shape[n, l] * sum_p poly[p+1, l] eps^p; poly: Matrix(degree+1, L) or nothing,
# shape: Matrix(N_T, L) or nothing
function set_amplitudes(h, poly::Union{Nothing,Matrix{Float64}}, shape::Union{Nothing,Matrix{Float64}})
    degree = poly === nothing ? 1 : size(poly, 1) - 1
    check(h, ccall((:krotov_set_amplitudes, lib), Cint, (Ptr{Cvoid}, Cint, Ptr{Float64}, Ptr{Float64}), h.ptr, degree,
                   poly === nothing ? C_NULL : pointer(poly), shape === nothing ? C_NULL : pointer(shape)))
end

# s[l] > 0: control l enters as shape[l][n] * poly_l(tanh(s[l] * eps)) (bounded amplitudes); `nothing` restores s = 0
function set_amplitude_saturation(h, s::Union{Nothing,Vector{Float64}})
    check(h, ccall((:krotov_set_amplitude_saturation, lib), Cint, (Ptr{Cvoid}, Ptr{Float64}), h.ptr,
                   s === nothing ? C_NULL : pointer(s)))
end

# control_of_term[t] (0-based control id of term t, numbered in order of first appearance) for a problem whose n_ctrl counts
# (operator, amplitude) terms; `nothing` = every term is its own control
function set_control_terms(h, control_of_term::Union{Nothing,Vector{Int32}})
    check(h, ccall((:krotov_set_control_terms, lib), Cint, (Ptr{Cvoid}, Ptr{Int32}), h.ptr,
                   control_of_term === nothing ? C_NULL : pointer(control_of_term)))
end

# pulses: Matrix{Float64}(N_T, L), column-major == [L][N_T] row-major on the wire
forward(h, pulses::Matrix{Float64}) =
    check(h, ccall((:krotov_forward, lib), Cint, (Ptr{Cvoid}, Ptr{Float64}), h.ptr, pulses))

# chi: Matrix{ComplexF64}(d, N) -- one column per trajectory
set_chi(h, chi::Matrix{ComplexF64}) =
    check(h, ccall((:krotov_set_chi, lib), Cint, (Ptr{Cvoid}, Ptr{Float64}), h.ptr, chi))

# chi_k(T) = coef[k] * target[k], formed on the device (several ranks: the caller did the global sum of tau)
set_chi_coeffs(h, coef::Vector{ComplexF64}) =
    check(h, ccall((:krotov_set_chi_coeffs, lib), Cint, (Ptr{Cvoid}, Ptr{Float64}), h.ptr, coef))

iterate!(h, guess::Matrix{Float64}, new::Matrix{Float64}, g_a_int::Vector{Float64}) =
    check(h, ccall((:krotov_iterate, lib), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                   h.ptr, guess, new, g_a_int))

get_states!(h, states::Matrix{ComplexF64}) =
    check(h, ccall((:krotov_get_states, lib), Cint, (Ptr{Cvoid}, Ptr{Float64}), h.ptr, states))

get_tau!(h, tau::Vector{ComplexF64}) =
    check(h, ccall((:krotov_get_tau, lib), Cint, (Ptr{Cvoid}, Ptr{Float64}), h.ptr, tau))

# columns n0:n1-1 (0-based grid index) of the storage of trajectory k (0-based); out: Matrix{ComplexF64}(d, n1 - n0)
get_storage!(h, which, k, n0, n1, out::Matrix{ComplexF64}) =
    check(h, ccall((:krotov_get_storage, lib), Cint, (Ptr{Cvoid}, Cint, Cint, Cint, Cint, Ptr{Float64}),
                   h.ptr, which, k, n0, n1, out))

function get_profile(h, cta::Integer = -1)
    out = Vector{Int64}(undef, 8)
    check(h, ccall((:krotov_get_profile, lib), Cint, (Ptr{Cvoid}, Cint, Ptr{Int64}), h.ptr, cta, out))
    out
end

# Multi-GPU (one Julia process per GPU): exchange the descriptors by any transport (MPI.Allgather, Distributed, ...),
# then connect; from then on `iterate!` exchanges the per-time-step overlap sums in-kernel over NVLink.
function comm_export(h)
    desc = Vector{UInt8}(undef, COMM_DESC_BYTES)
    check(h, ccall((:krotov_comm_export, lib), Cint, (Ptr{Cvoid}, Ptr{Cvoid}), h.ptr, desc))
    desc
end

# descs: Matrix{UInt8}(COMM_DESC_BYTES, world)
comm_connect(h, rank::Integer, world::Integer, descs::Matrix{UInt8}) =
    check(h, ccall((:krotov_comm_connect, lib), Cint, (Ptr{Cvoid}, Cint, Cint, Ptr{Cvoid}), h.ptr, rank, world, descs))

# several ranks emulated on one device (diagnostics): see include/krotov_cuda.h
function group_connect(hs::Vector{Handle})
    ptrs = Ptr{Cvoid}[h.ptr for h in hs]
    check(hs[1], ccall((:krotov_group_connect, lib), Cint, (Ptr{Ptr{Cvoid}}, Cint), ptrs, length(hs)))
end

function group_iterate!(hs::Vector{Handle}, guess::Matrix{Float64}, new::Array{Float64,3}, g_a_int::Matrix{Float64})
    ptrs = Ptr{Cvoid}[h.ptr for h in hs]
    check(hs[1], ccall((:krotov_group_iterate, lib), Cint, (Ptr{Ptr{Cvoid}}, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                       ptrs, length(hs), guess, new, g_a_int))
end

# Host utilities (pure host code in the same library; Julia's `eigvals` works unchanged).
# mats: Array{ComplexF64}(d, d, n_mat)
function hermitian_extremes(mats::Array{ComplexF64,3}; threads = 0)
    d, n = size(mats, 1), size(mats, 3)
    e_min, e_max = Vector{Float64}(undef, n), Vector{Float64}(undef, n)
    rc = ccall((:krotov_hermitian_extremes, lib), Cint, (Cint, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Cint),
               n, d, mats, e_min, e_max, threads)
    rc == 0 || error("libkrotov_cuda: krotov_hermitian_extremes: bad argument")
    e_min, e_max
end

# The envelope solved on the device from the terms the handle holds (persistent kernel path); amps: [L, n_corner]
function envelope_extremes_device(h::Handle, amps::Matrix{Float64}, n_gen::Integer)
    e_min, e_max = Vector{Float64}(undef, n_gen), Vector{Float64}(undef, n_gen)
    check(h, ccall((:krotov_envelope_extremes_device, lib), Cint, (Ptr{Cvoid}, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                   h.ptr, size(amps, 2), amps, e_min, e_max))
    e_min, e_max
end

# H0: [d, d, n_gen], Hc: [d, d, n_gen, L], amps: [L, n_corner]
function envelope_extremes(H0::Array{ComplexF64,3}, Hc::Array{ComplexF64,4}, amps::Matrix{Float64}; threads = 0)
    d, n_gen, L = size(H0, 1), size(H0, 3), size(Hc, 4)
    e_min, e_max = Vector{Float64}(undef, n_gen), Vector{Float64}(undef, n_gen)
    rc = ccall((:krotov_envelope_extremes, lib), Cint,
        (Cint, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Cint),
        n_gen, d, L, H0, Hc, size(amps, 2), amps, e_min, e_max, threads)
    rc == 0 || error("libkrotov_cuda: krotov_envelope_extremes: bad argument")
    e_min, e_max
end

end # module
