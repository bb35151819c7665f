# TorJCuda.jl — the ccall shim of INTEGRATION.md as a file a maintainer can `include` after src/plasma.jl.
# NOT EXECUTED in the build environment of this repository (Julia is not installed there); the same C ABI calls, in the
# same order, are exercised by the Python mirror torj_jl_b200/ and by tests/c_abi/abi_smoke.c.
# It replaces the bodies of abs_Al_init (reference src/absorption.jl:1-7), make_ray (src/solve.jl:135-181) and
# make_beam (src/solve.jl:209-242); Plasma(...) and launch_peripheral_rays stay as they are.

const libtorj = joinpath(@__DIR__, "..", "deps", "libtorj_cuda.so")

struct TorjOptions          # torj_options (include/torj_cuda.h, TORJ_ABI_VERSION 3), field for field
    scheme::Int32; n_segments::Int32
    dtmax::Float64; abstol::Float64; reltol::Float64; psi_stop::Float64; p_stop::Float64; te_min::Float64
    max_harmonic::Int32; max_steps_per_segment::Int32
    alpha_floor::Float64
    schedule::Int32; absorption_model::Int32; lanes_per_ray::Int32; reserved_::Int32
end
struct TorjGrid; nR::Int32; nZ::Int32; R_first::Float64; R_last::Float64; Z_first::Float64; Z_last::Float64; end
struct TorjCounters; n_acc::Int64; n_rej::Int64; n_rhs::Int64; n_alpha::Int64; n_harm::Int64; n_rays_ok::Int64; n_harm_pruned::Int64; n_alpha_skipped::Int64; end

torj_check(rc) = rc == 0 || error(unsafe_string(ccall((:torj_last_error, libtorj), Cstring, ())))

const _ctx = Ref{Ptr{Cvoid}}(C_NULL)
function torj_ctx()
    if _ctx[] == C_NULL
        @assert ccall((:torj_abi_version, libtorj), Cint, ()) == 3   # the struct layouts above are TORJ_ABI_VERSION 3
        torj_check(ccall((:torj_ctx_create, libtorj), Cint, (Cint, Ptr{Cvoid}, Ref{Ptr{Cvoid}}), 0, C_NULL, _ctx))
    end
    _ctx[]
end

# Exact deposition sums for every later call on this context (torj_ctx_set_exact_sum): dP_dV and deposited_power then
# come out bit-identical under any schedule, ray order and device count, like the reference's serial sum is run to run.
# Weights |w| <= 2^40. Off (false) is the default and today's floating-point atomics.
set_exact_sum!(on::Bool) = torj_check(ccall((:torj_ctx_set_exact_sum, libtorj), Cint, (Ptr{Cvoid}, Int32), torj_ctx(), Int32(on)))

# Options: the reference's hard-coded constants (torj_options_default) with keyword overrides, e.g.
# torj_options(absorption_model = 1) for the warm-plasma damping of src/general_absorption.jl.
function torj_options(; kw...)
    o = Ref{TorjOptions}()
    ccall((:torj_options_default, libtorj), Cvoid, (Ref{TorjOptions},), o)
    isempty(kw) && return o
    vals = Any[getfield(o[], k) for k in fieldnames(TorjOptions)]
    for (k, v) in kw
        i = findfirst(==(k), fieldnames(TorjOptions))
        i === nothing && throw(ArgumentError("torj_options has no field $k"))
        vals[i] = convert(fieldtype(TorjOptions, i), v)
    end
    Ref(TorjOptions(vals...))
end

# abs_Al_init(N)  — src/absorption.jl:1-7 keeps filling the Julia globals and additionally uploads them
function abs_Al_init(N_absz::Int)
    global _int_weights, _int_absz
    _int_absz, _int_weights = gausslegendre(N_absz)
    torj_check(ccall((:torj_abs_init, libtorj), Cint, (Ptr{Cvoid}, Int32, Ptr{Float64}, Ptr{Float64}),
                     torj_ctx(), N_absz, _int_absz, _int_weights))
end

# Device tables of a Plasma: created ONCE per Plasma object and destroyed with it. The handle lives in a mutable holder
# whose finalizer calls torj_plasma_destroy; the holder is kept in a WeakKeyDict keyed by the (immutable-content) Plasma,
# so it dies — and frees the 3.2 MB of tables — when the Plasma is garbage collected. (`Plasma` is a plain struct in the
# reference, src/plasma.jl:2-14; if it is not mutable, make it `mutable struct` or key the dict by `objectid`.)
mutable struct TorjPlasmaHandle
    ptr::Ptr{Cvoid}
    function TorjPlasmaHandle(ptr)
        h = new(ptr)
        finalizer(h) do x
            x.ptr == C_NULL || ccall((:torj_plasma_destroy, libtorj), Cvoid, (Ptr{Cvoid},), x.ptr)
            x.ptr = C_NULL
        end
        h
    end
end
const _plasmas = WeakKeyDict{Any,TorjPlasmaHandle}()

# Two routes to the tables:
#  (a) hand over the already prefiltered padded coefficient matrices of the six 2-D splines and the 1-D V(ψ) spline
#      (Extrapolation -> ScaledInterpolation -> BSplineInterpolation);
#  (b) if those Interpolations.jl internals move: keep the constructor's raw arrays and call torj_plasma_create_from_data
#      (1-D resampling/log/prefilter on the host, the six 2-D prefilters and the packing on the GPU) — the natural cubic
#      spline is unique, so the tables are the same to rounding.
coefs(spl) = Matrix{Float64}(parent(spl.itp.itp.coefs))
function torj_plasma(p::Plasma)
    get!(_plasmas, p) do
        g = TorjGrid(length(p.R_coords), length(p.Z_coords), p.R_coords[1], p.R_coords[end], p.Z_coords[1], p.Z_coords[end])
        vr = p.volume_psi_spline.itp.ranges[1]
        vc = Vector{Float64}(parent(p.volume_psi_spline.itp.itp.coefs))
        h = Ref{Ptr{Cvoid}}(C_NULL)
        torj_check(ccall((:torj_plasma_create, libtorj), Cint,
            (Ptr{Cvoid}, Ref{TorjGrid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
             Ptr{Float64}, Int32, Float64, Float64, Float64, Ref{Ptr{Cvoid}}),
            torj_ctx(), g, coefs(p.psi_norm_spline), coefs(p.ne_spline), coefs(p.Te_spline), coefs(p.Br_spline),
            coefs(p.Bz_spline), coefs(p.Bϕ_spline), vc, length(vr), first(vr), step(vr), p.psi_prof_max, h))
        TorjPlasmaHandle(h[])
    end.ptr
end

function torj_trace(hp, pos::Matrix{Float64}, dir::Matrix{Float64}, w::Vector{Float64}, f, mode, s_max, psi;
                    traj::UnitRange=1:0, max_pts=0, options=torj_options())
    n = length(w); npsi = length(psi); nt = length(traj)
    dP_dV = zeros(npsi); dep = Ref(0.0); Pf = zeros(n); Pd = zeros(n); npts = zeros(Int32, n); st = zeros(Int32, n)
    ts = zeros(max_pts, nt); txyz = zeros(max_pts, 3, nt); tP = zeros(max_pts, nt); tdP = zeros(max_pts, nt); tprof = zeros(npsi, nt)
    cnt = Ref{TorjCounters}()
    torj_check(ccall((:torj_trace, libtorj), Cint,
        (Ptr{Cvoid}, Ptr{Cvoid}, Ref{TorjOptions}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ref{Float64}, Ref{Int32}, Int32,
         Float64, Int32, Ptr{Float64}, Int32, Ptr{Int32}, Ptr{Float64}, Ref{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Ptr{Int32},
         Int64, Int64, Int32, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ref{TorjCounters}),
        torj_ctx(), hp, options, n, pos, dir, w, Float64(f), Int32(mode), 0, s_max, npsi, psi, 1, C_NULL, dP_dV, dep, Pf, Pd, npts, st,
        first(traj) - 1, nt, max_pts, ts, txyz, tP, tdP, tprof, cnt))
    (; dP_dV, deposited = dep[], Pf, Pd, npts, st, ts, txyz, tP, tdP, tprof, counters = cnt[])
end

# status 0 = OK, 3 = ended outside the (R,Z) grid (informational), 6 = trajectory buffer too small; the others are the
# reference's assertions (src/solve.jl:32,138,141) and the cut-off return (src/solve.jl:55-59)
ray_ok(st) = st == 0 || st == 3
max_points(s_max, o) = 2 + o[].n_segments * (ceil(Int, s_max / o[].n_segments / o[].dtmax) + 8)

# make_ray — src/solve.jl:135-181, same signature and return tuple
function make_ray(plasma::Plasma, x0, N_vacuum, f, mode::Integer, s_max::Float64, psi_dP_dV; options=torj_options())
    r = torj_trace(torj_plasma(plasma), reshape(collect(x0), 1, 3), reshape(collect(N_vacuum), 1, 3), [1.0], f, mode, s_max,
                   psi_dP_dV; traj=1:1, max_pts=max_points(s_max, options), options)
    ray_ok(r.st[1]) || throw(AssertionError("ray status $(r.st[1])"))     # src/solve.jl:32,138,141
    n = r.npts[1]
    return r.ts[1:n, 1], [r.txyz[i, :, 1] for i in 1:n], r.tP[1:n, 1], r.tprof[:, 1], r.Pd[1]
end

# make_beam — src/solve.jl:209-242: the Dagger.@spawn loop and the weighted reduction become one call
function make_beam(plasma::Plasma, r, phi, z, tor, pol, spot, invRc, f, mode::Integer, s_max::Float64, psi_dP_dV;
                   options=torj_options(), kwargs...)
    N0 = collect(IMAS.pol_tor_angles_2_vector(pol, tor)); x0 = [r * cos(phi), r * sin(phi), z]
    pos, dir, w = launch_peripheral_rays(x0, N0, spot, invRc, f; kwargs...)
    n = length(w)
    q = torj_trace(torj_plasma(plasma), pos, dir, w, f, mode, s_max, psi_dP_dV; traj=1:n,
                   max_pts=max_points(s_max, options), options)
    all(ray_ok, q.st) || throw(AssertionError("ray status $(q.st)"))
    arc = [q.ts[1:q.npts[i], i] for i in 1:n]
    traj = [[q.txyz[k, :, i] for k in 1:q.npts[i]] for i in 1:n]
    pw = [q.tP[1:q.npts[i], i] for i in 1:n]
    return arc, traj, pw, q.dP_dV, q.deposited, w
end

# make_beam_series — make_beam of one launcher on each plasma of a vector of plasmas on ONE (R,Z) grid (time slices, an
# equilibrium ensemble) in one call, torj_trace_plasmas: the beam's rays go in once per plasma, contiguous, beam k through
# plasmas[k] with its profile normalised by that plasma's V(psi). No trajectories. The plasmas' tables must outlive the call
# (they do: torj_plasma(p) keeps them with p). Returns (dP_dV[n_psi, n_plasmas], deposited_power[n_plasmas], ray_weights,
# P_final[n_rays, n_plasmas]).
function make_beam_series(plasmas::Vector, r, phi, z, tor, pol, spot, invRc, f, mode::Integer, s_max::Float64, psi_dP_dV;
                          options=torj_options(), kwargs...)
    N0 = collect(IMAS.pol_tor_angles_2_vector(pol, tor)); x0 = [r * cos(phi), r * sin(phi), z]
    pos, dir, w = launch_peripheral_rays(x0, N0, spot, invRc, f; kwargs...)
    n = length(w); K = length(plasmas); npsi = length(psi_dP_dV)
    hs = Ptr{Cvoid}[torj_plasma(p) for p in plasmas]
    beam = Int32.(repeat(0:K-1, inner=n)); bp = Int32.(collect(0:K-1))
    dP_dV = zeros(npsi, K); dep = zeros(K); Pf = zeros(n * K); Pd = zeros(n * K); npts = zeros(Int32, n * K); st = zeros(Int32, n * K)
    cnt = Ref{TorjCounters}()
    torj_check(ccall((:torj_trace_plasmas, libtorj), Cint,
        (Ptr{Cvoid}, Int32, Ptr{Ptr{Cvoid}}, Ptr{Int32}, Ref{TorjOptions}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ref{Float64},
         Ref{Int32}, Int32, Float64, Int32, Ptr{Float64}, Int32, Ptr{Int32}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
         Ptr{Int32}, Ptr{Int32}, Int64, Int64, Int32, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
         Ref{TorjCounters}),
        torj_ctx(), K, hs, bp, options, n * K, repeat(pos, K), repeat(dir, K), repeat(w, K), Float64(f), Int32(mode), 0, s_max,
        npsi, psi_dP_dV, K, beam, dP_dV, dep, Pf, Pd, npts, st, 0, 0, 0, C_NULL, C_NULL, C_NULL, C_NULL, C_NULL, cnt))
    all(ray_ok, st) || throw(AssertionError("ray status $(st)"))
    return dP_dV, dep, w, reshape(Pf, n, K)
end

# α(omega, X, Y, N_r, theta, te, v_g_perp, imod) — src/general_absorption.jl:1328-1337 on the device (no set_extv! needed)
function α(omega::Real, X::Real, Y::Real, N_r::Real, theta::Real, te::Real, v_g_perp::Real, imod::Integer)
    Nw = Ref(0.0); al = Ref(0.0); lrm = Ref(Int32(0)); ierr = Ref(Int32(0))
    torj_check(ccall((:torj_warm_alpha, libtorj), Cint,
        (Ptr{Cvoid}, Int64, Ref{Float64}, Ref{Float64}, Ref{Float64}, Ref{Float64}, Ref{Float64}, Ref{Float64}, Ref{Float64}, Int32,
         Ref{Float64}, Ref{Float64}, Ref{Int32}, Ref{Int32}),
        torj_ctx(), 1, Float64(omega), Float64(X), Float64(Y), Float64(N_r), Float64(theta), Float64(te), Float64(v_g_perp),
        Int32(imod), Nw, al, lrm, ierr))
    return Nw[], al[]
end

# ---- one process per GPU (MPI.jl + CUDA.jl): exact sums across ranks -------------------------------------------------
# After an exact-sum trace the bundle's integer accumulator is summed over the ranks word by word (MPI.Allreduce! of Int64
# with +), then converted once: dP_dV and the deposited power are the bits of one trace of every rank's rays, at a fixed
# lanes_per_ray. The agreement first (ok and the word count, MIN) makes every rank throw when one rank's trace failed or
# the lengths differ, instead of leaving the others waiting in the sum. This sketch needs n >= 1 rays on every rank.
exact_words(b) = (p = Ref{Ptr{Cvoid}}(C_NULL); n = Ref{Int64}(0);
                  torj_check(ccall((:torj_bundle_device_exact_words, libtorj), Cint, (Ptr{Cvoid}, Ref{Ptr{Cvoid}}, Ref{Int64}), b, p, n));
                  (p[], n[]))
finalize_exact!(b) = torj_check(ccall((:torj_bundle_finalize_exact, libtorj), Cint, (Ptr{Cvoid},), b))
function torj_trace_exact_mpi(hp, pos::Matrix{Float64}, dir::Matrix{Float64}, w::Vector{Float64}, f, mode, s_max, psi, comm;
                              options=torj_options())
    set_exact_sum!(true)
    n = length(w); npsi = length(psi); b = Ref{Ptr{Cvoid}}(C_NULL)
    dP_dV = zeros(npsi); dep = Ref(0.0); Pf = zeros(n); Pd = zeros(n); npts = zeros(Int32, n); st = zeros(Int32, n)
    try
        words, nw = C_NULL, 0
        try
            torj_check(ccall((:torj_bundle_create, libtorj), Cint, (Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
                Ref{Float64}, Ref{Int32}, Int32, Ref{Ptr{Cvoid}}), torj_ctx(), n, pos, dir, w, Float64(f), Int32(mode), 0, b))
            torj_check(ccall((:torj_bundle_trace, libtorj), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Ref{TorjOptions}, Float64, Int32,
                Ptr{Float64}), b[], hp, options, s_max, npsi, psi))
            words, nw = exact_words(b[])
        catch
            MPI.Allreduce(Int64[0, typemax(Int64), typemax(Int64)], min, comm)   # join the agreement as failed
            rethrow()
        end
        ok, lo, neg_hi = MPI.Allreduce(Int64[1, nw, -nw], min, comm)
        ok == 1 || error("torj_trace_exact_mpi: the trace failed on another rank")
        lo == -neg_hi || error("torj_trace_exact_mpi: the ranks' accumulators differ in length ($lo to $(-neg_hi) words)")
        torj_check(ccall((:torj_ctx_sync, libtorj), Cint, (Ptr{Cvoid},), torj_ctx()))
        buf = unsafe_wrap(CuArray, CuPtr{Int64}(UInt(words)), nw)   # the library's buffer, no copy (CUDA-aware MPI)
        MPI.Allreduce!(buf, +, comm)
        CUDA.synchronize()
        finalize_exact!(b[])
        torj_check(ccall((:torj_bundle_results, libtorj), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ref{Float64}, Ptr{Float64},
            Ptr{Float64}, Ptr{Int32}, Ptr{Int32}, Ptr{Cvoid}), b[], dP_dV, dep, Pf, Pd, npts, st, C_NULL))
    finally
        ccall((:torj_bundle_destroy, libtorj), Cvoid, (Ptr{Cvoid},), b[])
    end
    (; dP_dV, deposited = dep[], Pf, Pd, npts, st)
end

# ---- several GPUs from this one Julia process: bind torj_multi_* instead (same arguments as torj_trace) ---------------
# torj_multi_create opens every visible device and the NCCL communicators (ncclCommInitAll); torj_multi_trace shards the
# rays (contiguous, or beams dealt round-robin after torj_multi_configure(m, 1, rays_per_beam, 0)), traces every shard on
# its device and sums the profiles with ONE ncclAllReduce over NVLink on the devices' buffers.
const _multi = Ref{Ptr{Cvoid}}(C_NULL)
function torj_multi()
    if _multi[] == C_NULL
        torj_check(ccall((:torj_multi_create, libtorj), Cint, (Int32, Ref{Ptr{Cvoid}}), 0, _multi))
        atexit() do  # the per-device copies of the plasmas first: they live on the contexts of the torj_multi
            foreach(h -> ccall((:torj_multi_plasma_destroy, libtorj), Cvoid, (Ptr{Cvoid},), h), _mplasmas)
            empty!(_mplasmas)
            ccall((:torj_multi_destroy, libtorj), Cvoid, (Ptr{Cvoid},), _multi[])
        end
    end
    _multi[]
end

# Exact sums on every device of torj_multi() (torj_multi_set_exact_sum): the devices' integer accumulators are summed
# (ncclInt64 all-reduce or on the host) before one conversion, giving the bits of one device tracing the whole bundle.
multi_set_exact_sum!(on::Bool) =
    torj_check(ccall((:torj_multi_set_exact_sum, libtorj), Cint, (Ptr{Cvoid}, Int32), torj_multi(), Int32(on)))

# torj_mplasma: one plasma's tables on every device of torj_multi(), built there from the arrays of the Plasma constructor
# (src/plasma.jl:30-32: 2-D arrays [nR, nZ], profiles and the 1-D volume; route (b) above). Kept until the process exits.
const _mplasmas = Ptr{Cvoid}[]
function torj_mplasma(R, Z, psi_norm, psi_prof, ne, Te, BR, BZ, Bphi, psi1d, vol1d)
    m = torj_multi()
    g = TorjGrid(length(R), length(Z), R[1], R[end], Z[1], Z[end])
    h = Ref{Ptr{Cvoid}}(C_NULL)
    torj_check(ccall((:torj_multi_plasma_create_from_data, libtorj), Cint,
        (Ptr{Cvoid}, Ref{TorjGrid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Int32, Ptr{Float64}, Ptr{Float64},
         Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Int32, Ref{Ptr{Cvoid}}),
        m, g, Matrix{Float64}(psi_norm), Vector{Float64}(psi_prof), Vector{Float64}(ne), Vector{Float64}(Te), length(psi_prof),
        Matrix{Float64}(BR), Matrix{Float64}(BZ), Matrix{Float64}(Bphi), Vector{Float64}(psi1d), Vector{Float64}(vol1d),
        length(psi1d), h))
    push!(_mplasmas, h[])
    h[]
end

# make_beam_series on every GPU (torj_multi_trace_plasmas): the same call and result as make_beam_series above, with
# torj_mplasma handles for the plasmas. The beam on each plasma is a whole block of n rays, and block-cyclic sharding with
# block_rays = n deals whole plasmas round-robin over the devices; contiguous sharding is restored afterwards.
function multi_make_beam_series(mplasmas::Vector{Ptr{Cvoid}}, r, phi, z, tor, pol, spot, invRc, f, mode::Integer,
                                s_max::Float64, psi_dP_dV; options=torj_options(), kwargs...)
    N0 = collect(IMAS.pol_tor_angles_2_vector(pol, tor)); x0 = [r * cos(phi), r * sin(phi), z]
    pos, dir, w = launch_peripheral_rays(x0, N0, spot, invRc, f; kwargs...)
    n = length(w); K = length(mplasmas); npsi = length(psi_dP_dV)
    beam = Int32.(repeat(0:K-1, inner=n)); bp = Int32.(collect(0:K-1))
    dP_dV = zeros(npsi, K); dep = zeros(K); Pf = zeros(n * K); Pd = zeros(n * K); npts = zeros(Int32, n * K); st = zeros(Int32, n * K)
    cnt = Ref{TorjCounters}()
    m = torj_multi()
    torj_check(ccall((:torj_multi_configure, libtorj), Cint, (Ptr{Cvoid}, Int32, Int64, Int32), m, 1, n, 0))
    try
        torj_check(ccall((:torj_multi_trace_plasmas, libtorj), Cint,
            (Ptr{Cvoid}, Int32, Ptr{Ptr{Cvoid}}, Ptr{Int32}, Ref{TorjOptions}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
             Ref{Float64}, Ref{Int32}, Int32, Float64, Int32, Ptr{Float64}, Int32, Ptr{Int32}, Ptr{Float64}, Ptr{Float64},
             Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Ptr{Int32}, Int64, Int64, Int32, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
             Ptr{Float64}, Ptr{Float64}, Ref{TorjCounters}),
            m, K, mplasmas, bp, options, n * K, repeat(pos, K), repeat(dir, K), repeat(w, K), Float64(f), Int32(mode), 0, s_max,
            npsi, psi_dP_dV, K, beam, dP_dV, dep, Pf, Pd, npts, st, 0, 0, 0, C_NULL, C_NULL, C_NULL, C_NULL, C_NULL, cnt))
    finally
        torj_check(ccall((:torj_multi_configure, libtorj), Cint, (Ptr{Cvoid}, Int32, Int64, Int32), m, 0, 1, 0))
    end
    all(ray_ok, st) || throw(AssertionError("ray status $(st)"))
    return dP_dV, dep, w, reshape(Pf, n, K)
end
