# DiscretePOMPGPU.jl -- the reference-side binding a maintainer adds to DiscretePOMP.jl to route the particle-filter hot
# path through libdpomp.so (include/dpomp.h).  Self-contained: every function it calls is defined here, in the reference
# (module DiscretePOMP) or in Julia Base / LinearAlgebra / Distributions.
#
# UNTESTED in this repository: there is no Julia toolchain in the build image (SURVEY.md F3).  The same call sequences
# are exercised through the same C ABI by the Python host (discretepomp.jl_b200/*.py) and by tests/c_driver.c.
#
# Usage (inside module DiscretePOMP, after the includes of src/DiscretePOMP.jl:72-106):
#     include("DiscretePOMPGPU.jl")
# Exported signatures (src/DiscretePOMP.jl:59-67) do not change.  Re-bound, with identical signatures:
#     get_log_pdf_fn          src/hmm_particle_filter.jl:87-101
#     estimate_likelihood     src/hmm_particle_filter.jl:79-84
#     run_pibis               src/hmm_ibis.jl:12-135     (its three partial_log_likelihood! call sites, batched)
#     run_mbp_ibis            src/hmm_ibis.jl:140-244    (iterate_particle!, deepcopy, partial_model_based_proposal loops)
#     rs_systematic           src/hmm_resample.jl:44-62
# plus DpompComm for sharding theta-particles over several GPUs (one Julia process per GPU).

import LinearAlgebra
import Distributions
import Statistics
import Random

const LIBDPOMP = get(ENV, "LIBDPOMP", "libdpomp")
const DPOMP_RS_SYSTEMATIC, DPOMP_RS_STRATIFIED, DPOMP_RS_MULTINOMIAL = Int32(1), Int32(2), Int32(3)
const DPOMP_UNIQUE_ID_BYTES = 128
const DPOMP_OBS_GAUSSIAN, DPOMP_OBS_POISSON, DPOMP_OBS_BINOMIAL, DPOMP_OBS_NEGBIN = Int32(0), Int32(1), Int32(2), Int32(3)

# struct dpomp_model_desc (include/dpomp.h); NTuple-of-64 fields are the row-major [8][8] C arrays
struct DpompModelDesc
    n_compartments::Int32; n_events::Int32; n_params::Int32; t0_index::Int32
    rate_par::NTuple{8,Int32}
    rate_f1::NTuple{64,Int32}; rate_k1::NTuple{8,Int32}
    rate_f2::NTuple{64,Int32}; rate_k2::NTuple{8,Int32}
    rate_has_den::NTuple{8,Int32}
    rate_dn::NTuple{64,Int32}; rate_kd::NTuple{8,Int32}
    trans::NTuple{64,Int32}
    initial_condition::NTuple{8,Int64}
    obs_sigma::Float64
    obs_xmask::NTuple{8,Int32}
    n_obs_vals::Int32
    obs_ymask::NTuple{8,Int32}
    n_obs::Int32
    obs_time::Ptr{Float64}; obs_id::Ptr{Int32}; obs_val::Ptr{Int64}
end

struct ModelCompileError <: Exception
    msg::String
end
Base.showerror(io::IO, e::ModelCompileError) = print(io, "ModelCompileError: ", e.msg)

dpomp_check(rc) = rc == 0 ? nothing :
    error("libdpomp (", rc, "): ", unsafe_string(ccall((:dpomp_last_error, LIBDPOMP), Cstring, ())))

pad(v, n, T) = ntuple(i -> i <= length(v) ? T(v[i]) : zero(T), n)
pad(v, n, T, fill) = ntuple(i -> i <= length(v) ? T(v[i]) : T(fill), n)
rows(m::AbstractMatrix, T) = ntuple(k -> (e = (k - 1) ÷ 8 + 1; c = (k - 1) % 8 + 1;
                                          e <= size(m, 1) && c <= size(m, 2) ? T(m[e, c]) : zero(T)), 64)

# --------------------------------------------------------------------------------------------------------------------
# Model closures -> device rate table.  Closures cannot run on the device: the host PROBES rate_function / obs_model and
# fits    rate[e] = theta[p_e] * (k1 + f1.x) * (k2 + f2.x) / (kd + dn.x)      (small integer forms)
#         log g   = log(1/(sqrt(2 pi) sigma)) - (ymask.y - xmask.x)^2 / (2 sigma^2)
#                   or a Poisson / binomial / negative-binomial log pmf of Y = ymask.y given X = xmask.x (0/1 masks)
# which covers every predefined model (src/hmm_examples.jl:103-168 incl. freq_dep and ROSSMAC) and the custom model of
# test/runtests.jl:74-100; the fit is verified on random states and anything else throws ModelCompileError (there is no
# CPU fallback).  Same algorithm as discretepomp.jl_b200/rate_table.py (compile_rate_table / compile_obs_table), which
# is the tested implementation.
# --------------------------------------------------------------------------------------------------------------------
struct RateTable
    par::Vector{Int}            # 0-based parameter index or -1
    f1::Matrix{Int}; k1::Vector{Int}
    f2::Matrix{Int}; k2::Vector{Int}
    has_den::Vector{Int}; dn::Matrix{Int}; kd::Vector{Int}
end
struct ObsTable
    sigma::Float64
    xmask::Vector{Int}
    ymask::Vector{Int}
    family::Int32                 # DPOMP_OBS_*; count families: parameter i = theta[par_index[i] + 1] or, for -1, par_value[i]
    par_index::NTuple{2,Int32}    # 0-based (the C ABI's convention)
    par_value::NTuple{2,Float64}
end
ObsTable(sigma, xmask, ymask) = ObsTable(sigma, xmask, ymask, DPOMP_OBS_GAUSSIAN, (Int32(-1), Int32(-1)), (0.0, 0.0))

## log pmf of the count families with the boundary cases of include/dpomp.h (same association as rate_table.count_logpmf)
function count_logpmf(family, y::Integer, x::Integer, a::Float64, k::Float64 = 0.0)
    y < 0 && return -Inf
    yf, xf = Float64(y), Float64(x)
    if family == DPOMP_OBS_POISSON
        0.0 < a < Inf || return -Inf
        x == 0 && return y == 0 ? 0.0 : -Inf
        ylog = y == 0 ? 0.0 : yf * (log(a) + log(xf))
        return (ylog - a * xf) - lgamma_f64(yf + 1.0)
    elseif family == DPOMP_OBS_BINOMIAL
        (0.0 <= a <= 1.0 && y <= x) || return -Inf
        a == 0.0 && return y == 0 ? 0.0 : -Inf
        a == 1.0 && return y == x ? 0.0 : -Inf
        nx = xf - yf
        r = (lgamma_f64(xf + 1.0) - lgamma_f64(yf + 1.0)) - lgamma_f64(nx + 1.0)
        return (r + yf * log(a)) + nx * log1p(-a)
    else
        (0.0 < a < Inf && 0.0 < k < Inf) || return -Inf
        x == 0 && return y == 0 ? 0.0 : -Inf
        mu = a * xf; km = k + mu
        r = ((lgamma_f64(yf + k) - lgamma_f64(k)) - lgamma_f64(yf + 1.0)) + k * log(k / km)
        return y == 0 ? r : r + yf * log(mu / km)
    end
end
lgamma_f64(v::Float64) = Distributions.SpecialFunctions.logabsgamma(v)[1]

## count observation models with the reference's closure signature obs_model(y, population, theta); seq / y_seq are 1-based
## compartment / value indices, *_index a 1-based theta component (nothing = the fixed value)
struct CountObsModel <: Function
    family::Int32
    par_index::NTuple{2,Int32}
    par_value::NTuple{2,Float64}
    seq::Vector{Int}
    y_seq::Vector{Int}
end
function (m::CountObsModel)(y, population, theta)
    a, k = ntuple(i -> m.par_index[i] >= 0 ? Float64(theta[m.par_index[i] + 1]) : m.par_value[i], 2)
    return count_logpmf(m.family, sum(y.val[m.y_seq]), sum(population[m.seq]), a, k)
end
_idx(i) = i === nothing ? Int32(-1) : Int32(i - 1)
partial_poisson_obs_model(rho = 1.0; rho_index = nothing, seq = 2:2, y_seq = seq) =
    CountObsModel(DPOMP_OBS_POISSON, (_idx(rho_index), Int32(-1)), (Float64(rho), 0.0), collect(seq), collect(y_seq))
partial_binomial_obs_model(p = 1.0; p_index = nothing, seq = 2:2, y_seq = seq) =
    CountObsModel(DPOMP_OBS_BINOMIAL, (_idx(p_index), Int32(-1)), (Float64(p), 0.0), collect(seq), collect(y_seq))
partial_negbin_obs_model(rho = 1.0, k = 1.0; rho_index = nothing, k_index = nothing, seq = 2:2, y_seq = seq) =
    CountObsModel(DPOMP_OBS_NEGBIN, (_idx(rho_index), _idx(k_index)), (Float64(rho), Float64(k)), collect(seq), collect(y_seq))

function call_rates(rate_function::Function, E::Int, theta::Vector{Float64}, x::Vector{Int64})
    out = zeros(Float64, E)
    rate_function(out, theta, x)
    return out
end

# monomials 1, x_a, x_a x_b (a <= b) of a state
function monomials(x::Vector{Int64})
    C = length(x)
    out = Float64[1.0]
    append!(out, Float64.(x))
    for a in 1:C, b in a:C
        push!(out, Float64(x[a] * x[b]))
    end
    return out
end

# least-squares fit of an integer-coefficient quadratic polynomial; nothing if it does not fit
function fit_quadratic(points::Vector{Vector{Int64}}, vals::Vector{Float64}; tol = 1e-7)
    A = permutedims(hcat([monomials(p) for p in points]...))
    coef = A \ vals
    rounded = round.(coef)
    maximum(abs.(coef .- rounded)) > tol && return nothing
    maximum(abs.(A * rounded .- vals)) > tol * max(1.0, maximum(abs.(vals))) && return nothing
    return Int.(rounded)
end

function poly_of_forms(k1::Int, f1::Vector{Int}, k2::Int, f2::Vector{Int})
    C = length(f1)
    out = Int[k1 * k2]
    for a in 1:C
        push!(out, k1 * f2[a] + k2 * f1[a])
    end
    for a in 1:C, b in a:C
        push!(out, a == b ? f1[a] * f2[a] : f1[a] * f2[b] + f1[b] * f2[a])
    end
    return out
end

# write an integer quadratic polynomial as (k1 + f1.x)(k2 + f2.x) with 0/1 coefficients in L1; nothing if impossible
function factor_quadratic(poly::Vector{Int}, C::Int)
    lin = poly[2:(1 + C)]
    quad = poly[(2 + C):end]
    if all(quad .== 0)                                   # affine: L2 = 1
        return (poly[1], copy(lin), 1, zeros(Int, C))
    end
    qmat = zeros(Int, C, C)
    k = 1
    for a in 1:C, b in a:C
        qmat[a, b] = quad[k]; k += 1
    end
    for bits in Iterators.product(ntuple(_ -> 0:1, C + 1)...)
        k1 = bits[1]
        f1 = collect(Int, bits[2:end])
        any(f1 .!= 0) || continue
        a0 = findfirst(!=(0), f1)                        # x_a0^2 coefficient gives f2[a0]
        f2 = zeros(Int, C)
        f2[a0] = qmat[a0, a0]
        for b in 1:C
            b == a0 && continue
            lo, hi = min(a0, b), max(a0, b)
            f2[b] = qmat[lo, hi] - f1[b] * f2[a0]        # coefficient of x_a0 x_b = f1[a0] f2[b] + f1[b] f2[a0]
        end
        k2 = lin[a0] - k1 * f2[a0]
        if poly_of_forms(k1, f1, k2, f2) == poly
            # canonical order: the factor whose leading compartment has the lower index first, which is how the reference
            # writes its mass-action products (theta * x_a * x_b with a < b, src/hmm_examples.jl:107-154)
            if any(f2 .!= 0) && findfirst(!=(0), f2) < findfirst(!=(0), f1)
                return (k2, f2, k1, f1)
            end
            return (k1, f1, k2, f2)
        end
    end
    return nothing
end

function eval_rate_table(t::RateTable, theta::Vector{Float64}, x::Vector{Int64})
    E = length(t.par)
    out = zeros(Float64, E)
    for e in 1:E
        p = t.par[e] >= 0 ? theta[t.par[e] + 1] : 1.0
        l1 = Float64(t.k1[e] + sum(t.f1[e, :] .* x))
        l2 = Float64(t.k2[e] + sum(t.f2[e, :] .* x))
        r = (p * l1) * l2
        if t.has_den[e] != 0
            d = t.kd[e] + sum(t.dn[e, :] .* x)
            r = d == 0 ? 0.0 : r / Float64(d)
        end
        out[e] = r
    end
    return out
end

function fit_rate_table(rate_function::Function, E::Int, n_params::Int, C::Int)
    (1 <= C <= 8 && 1 <= E <= 8 && 1 <= n_params <= 16) ||
        throw(ModelCompileError("model size (C=$C, E=$E, n_theta=$n_params) exceeds the device table limits"))
    rng = Random.MersenneTwister(20261018)
    tab = RateTable(fill(-1, E), zeros(Int, E, C), zeros(Int, E), zeros(Int, E, C), ones(Int, E),
                    zeros(Int, E), zeros(Int, E, C), zeros(Int, E))
    theta0 = 0.5 .+ rand(rng, n_params)
    x0 = Int64.(rand(rng, 3:19, C))
    r0 = call_rates(rate_function, E, theta0, x0)
    # 1. which parameter multiplies each rate
    for e in 1:E
        r0[e] == 0.0 && throw(ModelCompileError("event $e: rate is zero at a strictly positive state; cannot probe"))
        hits = Int[]
        for p in 1:n_params
            th = copy(theta0); th[p] *= 2.0
            ratio = call_rates(rate_function, E, th, x0)[e] / r0[e]
            if abs(ratio - 2.0) < 1e-9
                push!(hits, p - 1)
            elseif abs(ratio - 1.0) > 1e-9
                throw(ModelCompileError("event $e: rate is not linear in theta[$p]"))
            end
        end
        length(hits) > 1 && throw(ModelCompileError("event $e: rate depends on more than one parameter"))
        tab.par[e] = isempty(hits) ? -1 : hits[1]
    end
    # 2. state dependence with the parameters set to one
    n_mono = 1 + C + C * (C + 1) ÷ 2
    pts = [Int64.(rand(rng, 1:11, C)) for _ in 1:(3 * n_mono + 8)]
    vals = [call_rates(rate_function, E, ones(n_params), p) for p in pts]
    dens = Any[nothing]
    for k in C:-1:2, idx in combinations_of(C, k)
        d = zeros(Int, C); d[idx] .= 1
        push!(dens, d)
    end
    for e in 1:E
        done = false
        for dn in dens
            scaled = [dn === nothing ? vals[i][e] : vals[i][e] * sum(dn .* pts[i]) for i in eachindex(pts)]
            poly = fit_quadratic(pts, scaled)
            poly === nothing && continue
            fac = factor_quadratic(poly, C)
            fac === nothing && continue
            tab.k1[e], tab.f1[e, :], tab.k2[e], tab.f2[e, :] = fac[1], fac[2], fac[3], fac[4]
            if dn !== nothing
                tab.has_den[e] = 1; tab.dn[e, :] = dn
            end
            done = true
            break
        end
        done || throw(ModelCompileError("event $e: rate is not of the form theta_p * L1(x) * L2(x) / D(x) with small integer forms"))
    end
    # 3. verify on fresh random points
    for _ in 1:64
        th = 0.01 .+ 1.99 .* rand(rng, n_params)
        x = Int64.(rand(rng, 1:199, C))
        want = call_rates(rate_function, E, th, x)
        got = eval_rate_table(tab, th, x)
        all(isapprox.(got, want; rtol = 1e-12, atol = 0.0)) ||
            throw(ModelCompileError("rate table verification failed at theta=$th, x=$x: $got vs $want"))
    end
    return tab
end

# all k-subsets of 1:n (lexicographic)
function combinations_of(n::Int, k::Int)
    out = Vector{Vector{Int}}()
    function rec(start, cur)
        if length(cur) == k
            push!(out, copy(cur)); return
        end
        for i in start:n
            push!(cur, i); rec(i + 1, cur); pop!(cur)
        end
    end
    rec(1, Int[])
    return out
end

function fit_obs_table(obs_model::Function, C::Int, V::Int, n_params::Int)
    if obs_model isa CountObsModel
        xm, ym = zeros(Int, C), zeros(Int, V)
        xm[obs_model.seq] .= 1; ym[obs_model.y_seq] .= 1
        return ObsTable(1.0, xm, ym, obs_model.family, obs_model.par_index, obs_model.par_value)
    end
    tab = try
        fit_gaussian_obs(obs_model, C, V, n_params)
    catch e
        e isa Union{DomainError, InexactError, OverflowError} || rethrow()
        nothing
    end
    tab === nothing && (tab = fit_count_obs(obs_model, C, V, n_params))
    tab === nothing && throw(ModelCompileError("obs_model is not a Gaussian in integer masks of (y, x), nor a Poisson, binomial or " *
                                               "negative-binomial law of 0/1 masks; no device table"))
    return tab
end

function fit_gaussian_obs(obs_model::Function, C::Int, V::Int, n_params::Int)
    theta = ones(n_params)
    g(yv, xv) = Float64(obs_model(Observation(0.0, 1, 1.0, Int64.(yv)), Int64.(xv), theta))
    zy, zx = zeros(Int64, V), zeros(Int64, C)
    a = g(zy, zx)
    sigma = exp(-a) / sqrt(2.0 * pi)
    b = 2.0 * sigma * sigma
    xm, ym = zeros(Int, C), zeros(Int, V)
    for i in 1:C
        x = copy(zx); x[i] = 1
        xm[i] = Int(round(sqrt(max(0.0, (a - g(zy, x)) * b))))
    end
    for j in 1:V
        y = copy(zy); y[j] = 1
        ym[j] = Int(round(sqrt(max(0.0, (a - g(y, zx)) * b))))
    end
    function fix_signs!(mask, probe)                     # relative signs from pairwise probes: (m_i + s m_j)^2
        nz = findall(!=(0), mask)
        for i in nz[2:end]
            z = zeros(Int64, length(mask)); z[nz[1]] = 1; z[i] = 1
            abs((a - probe(z)) * b - (mask[nz[1]] + mask[i])^2) > 1e-6 && (mask[i] = -mask[i])
        end
    end
    fix_signs!(xm, z -> g(zy, z))
    fix_signs!(ym, z -> g(z, zx))
    rng = Random.MersenneTwister(7)
    tmp1, tmp2 = log(1.0 / (sqrt(2.0 * pi) * sigma)), 2.0 * sigma * sigma
    for _ in 1:64
        y = Int64.(rand(rng, 0:49, V)); x = Int64.(rand(rng, 0:49, C))
        d = sum(ym .* y) - sum(xm .* x)
        isapprox(tmp1 - d * d / tmp2, g(y, x); rtol = 1e-10, atol = 1e-12) || return nothing
    end
    return ObsTable(sigma, xm, ym)
end

snap(v) = (s = round(v; sigdigits = 12); abs(s - v) <= 1e-12 * abs(v) ? s : v)

## count-law probe, as rate_table._fit_count_obs: 0/1 masks from the components that move the value, parameters from probe
## points (g(0, X) = -rho X; g(1, 1) = log p; g(1, X) - g(0, X) = log(k mu / (k + mu)) at X = 1, 2), theta-indexing by
## perturbing each theta component, then 64 random verification points
function fit_count_obs(obs_model::Function, C::Int, V::Int, n_params::Int)
    rng = Random.MersenneTwister(11)
    theta0 = 0.2 .+ 0.6 .* rand(rng, n_params)
    g(yv, xv, th) = Float64(obs_model(Observation(0.0, 1, 1.0, Int64.(yv)), Int64.(xv), th))
    try
        x0, y0 = fill(Int64(50), C), ones(Int64, V)
        base = g(y0, x0, theta0)
        isfinite(base) || return nothing
        xm = [Int(g(y0, (x = copy(x0); x[i] += 1; x), theta0) != base) for i in 1:C]
        ym = [Int(g((y = copy(y0); y[j] += 1; y), x0, theta0) != base) for j in 1:V]
        (any(xm .== 1) && any(ym .== 1)) || return nothing
        ix, iy = findfirst(==(1), xm), findfirst(==(1), ym)
        G(yy, xx, th) = g((y = zeros(Int64, V); y[iy] = yy; y), (x = zeros(Int64, C); x[ix] = xx; x), th)
        function fit(family, th)
            family == DPOMP_OBS_POISSON && return (-G(0, 1, th), 0.0)
            family == DPOMP_OBS_BINOMIAL && return (exp(G(1, 1, th)), 0.0)
            e1 = exp(-(G(1, 1, th) - G(0, 1, th))); e2 = exp(-(G(1, 2, th) - G(0, 2, th)))
            return (1.0 / (2.0 * (e1 - e2)), 1.0 / (2.0 * e2 - e1))
        end
        for family in (DPOMP_OBS_POISSON, DPOMP_OBS_BINOMIAL, DPOMP_OBS_NEGBIN)
            n_par = family == DPOMP_OBS_NEGBIN ? 2 : 1
            vals = fit(family, theta0)
            all(isfinite, vals[1:n_par]) || continue
            idx, fixed = [Int32(-1), Int32(-1)], [0.0, 0.0]
            for i in 1:n_par
                for j in 1:n_params
                    isapprox(vals[i], theta0[j]; rtol = 1e-9) || continue
                    th = copy(theta0); th[j] *= 0.9
                    if isapprox(fit(family, th)[i], th[j]; rtol = 1e-9)
                        idx[i] = Int32(j - 1); break
                    end
                end
                idx[i] < 0 && (fixed[i] = snap(vals[i]))
            end
            tab = ObsTable(1.0, xm, ym, family, (idx[1], idx[2]), (fixed[1], fixed[2]))
            vrng = Random.MersenneTwister(7)
            ok = all(1:64) do _
                y = Int64.(rand(vrng, 0:19, V)); x = Int64.(rand(vrng, 0:59, C)); th = 0.2 .+ 0.6 .* rand(vrng, n_params)
                a, k = ntuple(i -> tab.par_index[i] >= 0 ? th[tab.par_index[i] + 1] : tab.par_value[i], 2)
                got, want = count_logpmf(family, sum(ym .* y), sum(xm .* x), a, k), g(y, x, th)
                got == want || isapprox(got, want; rtol = 1e-9, atol = 1e-9)
            end
            ok && return tab
        end
    catch e
        e isa Union{DomainError, InexactError, OverflowError, ArgumentError, BoundsError} || rethrow()
    end
    return nothing
end

# --------------------------------------------------------------------------------------------------------------------
# Handles (finalizers release the device memory)
# --------------------------------------------------------------------------------------------------------------------
mutable struct DpompModel
    handle::Ptr{Cvoid}
    n_params::Int
end

## replaces get_private_model's role for the device (src/DiscretePOMP.jl:96-99): closures -> tables -> dpomp_model
function dpomp_model(model::HiddenMarkovModel)
    ic = model.fn_initial_condition()
    E, C = model.n_events, length(ic)
    n_params = length(model.prior)
    tm = vcat([reshape(model.fn_transition(e), 1, C) for e in 1:E]...)      # rows = events
    rt = fit_rate_table(model.rate_function, E, n_params, C)
    V = length(model.obs_data[1].val)
    ot = fit_obs_table(model.obs_model, C, V, n_params)
    times = Float64[y.time for y in model.obs_data]
    ids = Int32[y.obs_id for y in model.obs_data]
    vals = Int64[y.val[v] for y in model.obs_data for v in 1:V]             # row t = y[t].val
    handle = Ref{Ptr{Cvoid}}(C_NULL)
    GC.@preserve times ids vals begin
        desc = DpompModelDesc(C, E, n_params, model.t0_index,
            pad(rt.par, 8, Int32, -1), rows(rt.f1, Int32), pad(rt.k1, 8, Int32), rows(rt.f2, Int32), pad(rt.k2, 8, Int32),
            pad(rt.has_den, 8, Int32), rows(rt.dn, Int32), pad(rt.kd, 8, Int32), rows(tm, Int32), pad(ic, 8, Int64),
            ot.sigma, pad(ot.xmask, 8, Int32), V, pad(ot.ymask, 8, Int32),
            length(times), pointer(times), pointer(ids), pointer(vals))
        dpomp_check(ccall((:dpomp_model_create, LIBDPOMP), Cint, (Ref{DpompModelDesc}, Ref{Ptr{Cvoid}}), desc, handle))
    end
    if ot.family != DPOMP_OBS_GAUSSIAN
        pidx, pval = Int32[ot.par_index...], Float64[ot.par_value...]
        rc = GC.@preserve pidx pval ccall((:dpomp_model_set_obs_model, LIBDPOMP), Cint, (Ptr{Cvoid}, Int32, Ptr{Int32}, Ptr{Float64}),
                                          handle[], ot.family, pidx, pval)
        rc == 0 || ccall((:dpomp_model_destroy, LIBDPOMP), Cint, (Ptr{Cvoid},), handle[])
        dpomp_check(rc)
    end
    m = DpompModel(handle[], n_params)      # the library copied the observations
    finalizer(x -> ccall((:dpomp_model_destroy, LIBDPOMP), Cint, (Ptr{Cvoid},), x.handle), m)
    return m
end

mutable struct DpompPF
    handle::Ptr{Cvoid}
    model::DpompModel        # keeps the model handle alive as long as the filter
    n_batch::Int
end
function DpompPF(mdl::DpompModel, n_particles, n_batch, rs_type; seed = rand(UInt64), device = -1)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    dpomp_check(ccall((:dpomp_pf_create, LIBDPOMP), Cint, (Ptr{Cvoid}, Int64, Int32, Int32, UInt64, Int32, Ref{Ptr{Cvoid}}),
                      mdl.handle, n_particles, n_batch, rs_type, seed, device, h))
    pf = DpompPF(h[], mdl, n_batch)
    finalizer(p -> ccall((:dpomp_pf_destroy, LIBDPOMP), Cint, (Ptr{Cvoid},), p.handle), pf)
    return pf
end
set_batch_offset!(pf::DpompPF, off) = dpomp_check(ccall((:dpomp_pf_set_batch_offset, LIBDPOMP), Cint, (Ptr{Cvoid}, Int64), pf.handle, off))
function set_filter_ids!(pf::DpompPF, ids::Vector{Int64})      # 0-based GLOBAL ids of the first length(ids) filters
    GC.@preserve ids dpomp_check(ccall((:dpomp_pf_set_filter_ids, LIBDPOMP), Cint, (Ptr{Cvoid}, Ptr{Int64}, Int32), pf.handle, ids, length(ids)))
end

## replaces estimate_likelihood (src/hmm_particle_filter.jl:79-84); fn_rs / essc are accepted for signature compatibility
function estimate_likelihood(model::HiddenMarkovModel, parameters::Array{Float64,1}, particles::Int64, pop_size::Int64, fn_rs::Function, essc::Float64)
    pf = DpompPF(dpomp_model(model), particles, 1, DPOMP_RS_SYSTEMATIC)
    out = Ref{Float64}(0.0)
    GC.@preserve parameters dpomp_check(ccall((:dpomp_pf_loglik, LIBDPOMP), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Int32, Ref{Float64}), pf.handle, parameters, 1, out))
    return out[]
end

## replaces get_log_pdf_fn (src/hmm_particle_filter.jl:87-101): same signature, same closure type
function get_log_pdf_fn(mdl::HiddenMarkovModel, p::Int64 = C_DF_PF_P, rs_type::Int64 = 1; essc::Float64 = C_DF_ESS_CRIT)
    pf = DpompPF(dpomp_model(mdl), p, 1, rs_type in (2, 3) ? Int32(rs_type) : DPOMP_RS_SYSTEMATIC)
    function comp_log_pdf(parameters::Array{Float64, 1})
        out = Ref{Float64}(0.0)
        GC.@preserve parameters dpomp_check(ccall((:dpomp_pf_loglik, LIBDPOMP), Cint,
            (Ptr{Cvoid}, Ptr{Float64}, Int32, Ref{Float64}), pf.handle, parameters, 1, out))
        return out[]
    end
    return comp_log_pdf
end

## the loop `for p in eachindex(pop): gx[p] = partial_log_likelihood!(pop[p], ...)` (src/hmm_ibis.jl:53-56):
## theta is the n_theta x B matrix, column-major = one theta vector per filter
function partial_log_likelihood_batch!(pf::DpompPF, theta::Array{Float64, 2}, ymin::Int64, ymax::Int64)
    gx = Array{Float64, 1}(undef, size(theta, 2))
    GC.@preserve theta gx dpomp_check(ccall((:dpomp_pf_partial, LIBDPOMP), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Int32, Int32, Int32, Ptr{Float64}), pf.handle, theta, size(theta, 2), ymin, ymax, gx))
    return gx
end

## `pop2[p] .= pop[nidx[p]]` (src/hmm_ibis.jl:74) and `pop[p] .= pop_f` (:108)
permute_filters!(pf::DpompPF, nidx::Array{Int64, 1}) =
    GC.@preserve nidx dpomp_check(ccall((:dpomp_pf_permute, LIBDPOMP), Cint, (Ptr{Cvoid}, Ptr{Int64}, Int32), pf.handle, nidx, length(nidx)))
copy_filters!(dst::DpompPF, src::DpompPF, dst_slots::Array{Int64, 1}, src_slots::Array{Int64, 1}) =
    isempty(dst_slots) ? nothing : GC.@preserve dst_slots src_slots dpomp_check(ccall((:dpomp_pf_copy_filters, LIBDPOMP), Cint,
        (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Int64}, Ptr{Int64}, Int32), dst.handle, src.handle, dst_slots, src_slots, length(dst_slots)))

## replaces rs_systematic (src/hmm_resample.jl:44-62): same return type (1-based Vector{Int64}); the search runs on the GPU
function rs_systematic(w::Array{Float64, 1})
    out = Array{Int64, 1}(undef, length(w)); u = [rand()]
    GC.@preserve w u out dpomp_check(ccall((:dpomp_resample_indices, LIBDPOMP), Cint,
        (Int32, Int32, Ptr{Float64}, Int64, Ptr{Float64}, Int64, Int64, Ptr{Int64}, Int32), 1, 0, w, length(w), u, 1, length(w), out, -1))
    return out
end

# --------------------------------------------------------------------------------------------------------------------
# Multi-GPU: one Julia process per GPU (Distributed / MPI.jl launch); theta-particles partitioned contiguously.  Rank 0
# draws the NCCL unique id, the host broadcasts its 128 bytes by whatever means it has, every rank creates the
# communicator.  DpompComm(nothing, 0, 1) is the single-process communicator (no NCCL).
# --------------------------------------------------------------------------------------------------------------------
mutable struct DpompComm
    handle::Ptr{Cvoid}
    rank::Int
    world::Int
end
function dpomp_unique_id()
    id = zeros(UInt8, DPOMP_UNIQUE_ID_BYTES)
    GC.@preserve id dpomp_check(ccall((:dpomp_comm_unique_id, LIBDPOMP), Cint, (Ptr{UInt8}, Int32), id, length(id)))
    return id
end
function DpompComm(id::Union{Nothing, Vector{UInt8}}, rank::Int, world::Int; device = -1)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    if id === nothing
        dpomp_check(ccall((:dpomp_comm_create, LIBDPOMP), Cint, (Ptr{UInt8}, Int32, Int32, Int32, Int32, Ref{Ptr{Cvoid}}), C_NULL, 0, rank, world, device, h))
    else
        GC.@preserve id dpomp_check(ccall((:dpomp_comm_create, LIBDPOMP), Cint, (Ptr{UInt8}, Int32, Int32, Int32, Int32, Ref{Ptr{Cvoid}}), id, length(id), rank, world, device, h))
    end
    c = DpompComm(h[], rank, world)
    finalizer(x -> ccall((:dpomp_comm_destroy, LIBDPOMP), Cint, (Ptr{Cvoid},), x.handle), c)
    return c
end
function partition_bounds(n::Int, comm::DpompComm)          # 1-based inclusive block lo:hi of this rank
    lo, hi = Ref{Int64}(0), Ref{Int64}(0)
    dpomp_check(ccall((:dpomp_partition_bounds, LIBDPOMP), Cint, (Int64, Int32, Int32, Ref{Int64}, Ref{Int64}), n, comm.world, comm.rank, lo, hi))
    return (lo[] + 1):hi[]
end
function allgather_rows(comm::DpompComm, local_rows::Array{Float64}, n_total::Int, width::Int)
    out = width == 1 ? Array{Float64,1}(undef, n_total) : Array{Float64,2}(undef, width, n_total)   # column = item
    GC.@preserve local_rows out dpomp_check(ccall((:dpomp_comm_allgather_f64, LIBDPOMP), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Int32, Ptr{Float64}), comm.handle, local_rows, n_total, width, out))
    return out
end
function partial_log_likelihood_allgather!(pf::DpompPF, comm::DpompComm, theta_local::Array{Float64,2}, ymin::Int64, ymax::Int64, n_total::Int)
    gx = Array{Float64,1}(undef, n_total)
    GC.@preserve theta_local gx dpomp_check(ccall((:dpomp_pf_partial_allgather, LIBDPOMP), Cint,
        (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float64}, Int32, Int32, Int32, Int64, Ptr{Float64}),
        pf.handle, comm.handle, theta_local, size(theta_local, 2), ymin, ymax, n_total, gx))
    return gx
end
resample_migrate!(pf::DpompPF, comm::DpompComm, nidx::Array{Int64,1}) =
    GC.@preserve nidx dpomp_check(ccall((:dpomp_pf_resample_migrate, LIBDPOMP), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Int64}, Int64),
                                        pf.handle, comm.handle, nidx, length(nidx)))

const DPOMP_COMM = Ref{DpompComm}()         # set by the launcher; defaults to the single-process communicator
dpomp_comm() = isassigned(DPOMP_COMM) ? DPOMP_COMM[] : (DPOMP_COMM[] = DpompComm(nothing, 0, 1))

# --------------------------------------------------------------------------------------------------------------------
# run_pibis (src/hmm_ibis.jl:12-135), same signature and return value.  The per-theta-particle loops become batched
# calls over this rank's block; theta, weights and every host decision are replicated on all ranks (same RNG seed), so
# the only exchanges are the all-gather of the increments and the migration of resampled populations.
# Stated departure: the mutation sweep proposes for all theta-particles at once, so the random-walk scale tj (only used
# when ind_prop = false) is frozen within a sweep and updated afterwards with the same factors.
# --------------------------------------------------------------------------------------------------------------------
function run_pibis(model::HiddenMarkovModel, theta::Array{Float64, 2}, ess_rs_crit::Float64, ind_prop::Bool, alpha::Float64, np::Int64; n_props = 1)
    comm = dpomp_comm()
    outer_p = size(theta, 2)
    start_time = time_ns()
    blk = partition_bounds(outer_p, comm)
    n_loc = length(blk)
    ess_crit = ess_rs_crit * outer_p
    theta = copy(theta)
    w = ones(outer_p)
    aw = [Distributions.logpdf(model.prior, theta[:, i]) for i in 1:outer_p]
    dm = dpomp_model(model)
    pf = DpompPF(dm, np, max(n_loc, 1), DPOMP_RS_SYSTEMATIC)          # resident filters of this rank's theta-particles
    pf_f = DpompPF(dm, np, max(n_loc, 1), DPOMP_RS_SYSTEMATIC)        # proposal filters
    set_batch_offset!(pf, first(blk) - 1)
    mu = zeros(size(theta, 1))
    cv = zeros(size(theta, 1), size(theta, 1))
    k_log = zeros(Int64, 2)
    bme = zeros(2)
    propd = Distributions.MvNormal(Matrix{Float64}(LinearAlgebra.I, size(theta, 1), size(theta, 1)))
    tj = 0.2
    obs_min = 1
    for obs_i in eachindex(model.obs_data)
        if model.obs_data[obs_i].obs_id > 0
            gx = partial_log_likelihood_allgather!(pf, comm, theta[:, blk], obs_min, obs_i, outer_p)      # :53-56
            aw .+= gx
            gx .= exp.(gx)
            lml = log(sum(w .* gx) / sum(w))
            bme[1] += lml
            w .*= gx
            compute_is_mu_covar!(mu, cv, theta, w)
            if compute_ess(w) < ess_crit
                propd = get_prop_density(cv, propd)
                nidx = rs_systematic(w)
                theta = theta[:, nidx]
                aw = aw[nidx]
                resample_migrate!(pf, comm, nidx)                                                         # :71-79
                mlr = Statistics.mean(gx[nidx]) * exp(lml)
                k_log[1] += outer_p
                mtd_gx = gx[nidx]
                for mki in 1:n_props                                                                      # :83-116, one sweep
                    theta_f = similar(theta)
                    for p in 1:outer_p
                        theta_f[:, p] = ind_prop ? get_mv_param(propd, 1.0, mu) : get_mv_param(propd, tj, theta[:, p])
                    end
                    prtf = [Distributions.logpdf(model.prior, theta_f[:, p]) for p in 1:outer_p]
                    mine = [p for p in blk if prtf[p] != -Inf]                                            # valid proposals of this rank
                    loc = zeros(2, n_loc)                                                                  # rows: aw_f, gx_f
                    if !isempty(mine)
                        set_filter_ids!(pf_f, Int64.(mine .- 1))
                        thf = theta_f[:, mine]
                        if obs_i == 1
                            g = partial_log_likelihood_batch!(pf_f, thf, 1, 1)
                            a = copy(g)
                        else
                            a = partial_log_likelihood_batch!(pf_f, thf, 1, obs_i - 1)
                            g = partial_log_likelihood_batch!(pf_f, thf, obs_i, obs_i)
                            a .+= g
                        end
                        loc[1, mine .- (first(blk) - 1)] = a
                        loc[2, mine .- (first(blk) - 1)] = g
                    end
                    all_fg = allgather_rows(comm, loc, outer_p, 2)
                    aw_f = all_fg[1, :] .+ [prtf[p] == -Inf ? 0.0 : prtf[p] for p in 1:outer_p]
                    gx_f = all_fg[2, :]
                    u = rand(outer_p)
                    accepted = [prtf[p] != -Inf && exp(aw_f[p] - aw[p]) > u[p] for p in 1:outer_p]       # :104
                    acc_mine = [p for p in mine if accepted[p]]
                    src = Int64[findfirst(==(p), mine) for p in acc_mine]
                    copy_filters!(pf, pf_f, Int64.(acc_mine .- (first(blk) - 1)), src)                     # :108
                    for p in 1:outer_p
                        if accepted[p]
                            mtd_gx[p] = exp(gx_f[p]); theta[:, p] = theta_f[:, p]; aw[p] = aw_f[p]
                        end
                    end
                    n_acc = count(accepted); n_rej = count(prtf .!= -Inf) - n_acc
                    k_log[2] += n_acc
                    tj *= alpha^n_acc * 0.999^n_rej
                end
                bme[2] += log(mlr / Statistics.mean(mtd_gx))
                w .= 1
            else
                bme[2] += log(sum(w .* gx) / sum(w))
            end
            obs_min = obs_i + 1
        end
    end
    compute_is_mu_covar!(mu, cv, theta, w)
    output = ImportanceSample(mu, cv, theta, w, time_ns() - start_time, -bme)
    comm.rank == 0 && println("- finished in ", print_runtime(output.run_time), " (AR = ", round(100.0 * k_log[2] / k_log[1]; sigdigits = 3), "%)")
    return output
end

# --------------------------------------------------------------------------------------------------------------------
# run_mbp_ibis (src/hmm_ibis.jl:140-244): each theta-particle is one trajectory in the device store (dpomp_mbp)
# --------------------------------------------------------------------------------------------------------------------
mutable struct DpompMBP
    handle::Ptr{Cvoid}
    model::DpompModel
    n::Int
end
# max_traj plays MAX_TRAJ (src/DiscretePOMP.jl:40); the store reserves max_traj events per trajectory, so the default is
# 8192 (a trajectory that overflows gets log-likelihood -Inf exactly like the reference's MAX_TRAJ guard, src/hmm_sim.jl:17-20)
function DpompMBP(mdl::DpompModel, n_particles; max_traj = min(MAX_TRAJ, 8192), seed = rand(UInt64), device = -1)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    dpomp_check(ccall((:dpomp_mbp_create, LIBDPOMP), Cint, (Ptr{Cvoid}, Int32, Int32, UInt64, Int32, Ref{Ptr{Cvoid}}),
                      mdl.handle, n_particles, max_traj, seed, device, h))
    s = DpompMBP(h[], mdl, n_particles)
    finalizer(x -> ccall((:dpomp_mbp_destroy, LIBDPOMP), Cint, (Ptr{Cvoid},), x.handle), s)
    return s
end
function mbp_iterate!(s::DpompMBP, theta::Array{Float64,2}, obs_i::Int, fresh::Bool)      # iterate_particle! (src/hmm_sim.jl:6-25)
    out = Array{Float64,1}(undef, size(theta, 2))
    GC.@preserve theta out dpomp_check(ccall((:dpomp_mbp_iterate, LIBDPOMP), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Int32, Int32, Int32, Ptr{Float64}), s.handle, theta, size(theta, 2), obs_i, fresh ? 1 : 0, out))
    return out
end
function mbp_propose!(s::DpompMBP, theta_i::Array{Float64,2}, theta_f::Array{Float64,2}, valid::Vector{UInt8}, ymax::Int)   # src/hmm_mbp.jl:83-108
    out = Array{Float64,2}(undef, 2, size(theta_i, 2))                                       # column p = log_like[1:2] of proposal p
    GC.@preserve theta_i theta_f valid out dpomp_check(ccall((:dpomp_mbp_propose, LIBDPOMP), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{UInt8}, Int32, Int32, Ptr{Float64}), s.handle, theta_i, theta_f, valid, size(theta_i, 2), ymax, out))
    return out
end
mbp_accept!(s::DpompMBP, slots::Vector{Int64}) = isempty(slots) ? nothing :
    GC.@preserve slots dpomp_check(ccall((:dpomp_mbp_accept, LIBDPOMP), Cint, (Ptr{Cvoid}, Ptr{Int64}, Int32), s.handle, slots, length(slots)))
mbp_resample_migrate!(s::DpompMBP, comm::DpompComm, nidx::Vector{Int64}) =
    GC.@preserve nidx dpomp_check(ccall((:dpomp_mbp_resample_migrate, LIBDPOMP), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Int64}, Int64),
                                        s.handle, comm.handle, nidx, length(nidx)))

function run_mbp_ibis(model::HiddenMarkovModel, theta::Array{Float64, 2}, ess_rs_crit::Float64, n_props::Int64, ind_prop::Bool, alpha::Float64, msgs::Bool = true)
    comm = dpomp_comm()
    outer_p = size(theta, 2)
    comm.rank == 0 && println("Running: ", outer_p, "-particle MBP-IBIS analysis (model: ", model.model_name, ")")
    start_time = time_ns()
    blk = partition_bounds(outer_p, comm)
    n_loc = length(blk)
    ess_crit = ess_rs_crit * outer_p
    theta = copy(theta)
    store = DpompMBP(dpomp_model(model), max(n_loc, 1))
    dpomp_check(ccall((:dpomp_mbp_set_batch_offset, LIBDPOMP), Cint, (Ptr{Cvoid}, Int64), store.handle, first(blk) - 1))
    prior = [Distributions.logpdf(model.prior, theta[:, p]) for p in 1:outer_p]                # Particle.prior (:153)
    log_like = zeros(outer_p)                                                                   # Particle.log_like[1]
    propd = Distributions.MvNormal(Matrix{Float64}(LinearAlgebra.I, size(theta, 1), size(theta, 1)))
    tj = 0.2
    w = ones(outer_p)
    mu = zeros(size(theta, 1))
    cv = zeros(size(theta, 1), size(theta, 1))
    k_log = zeros(Int64, 2)
    bme = zeros(2)
    for obs_i in eachindex(model.obs_data)
        lg_loc = n_loc > 0 ? mbp_iterate!(store, theta[:, blk], obs_i, obs_i == 1) : Float64[]      # :176-179
        lg = allgather_rows(comm, lg_loc, outer_p, 1)
        if model.obs_data[obs_i].obs_id > 0
            log_like .+= lg
            gx = exp.(lg)
            lml = log(sum(w .* gx) / sum(w))
            bme[1] += lml
            w .*= gx
            compute_is_mu_covar!(mu, cv, theta, w)
            if compute_ess(w) < ess_crit
                propd = get_prop_density(cv, propd)
                nidx = rs_systematic(w)
                mtd_gx = gx[nidx]
                mbp_resample_migrate!(store, comm, nidx)                                            # :196-199
                theta = theta[:, nidx]; prior = prior[nidx]; log_like = log_like[nidx]
                mlr = Statistics.mean(gx[nidx]) * exp(lml)
                k_log[1] += outer_p * n_props
                for mki in 1:n_props                                                                # :203-219, one sweep
                    theta_f = similar(theta)
                    for p in 1:outer_p
                        theta_f[:, p] = ind_prop ? get_mv_param(propd, 1.0, mu) : get_mv_param(propd, tj, theta[:, p])
                    end
                    prior_f = [Distributions.logpdf(model.prior, theta_f[:, p]) for p in 1:outer_p]
                    valid = UInt8[prior_f[p] != -Inf ? 1 : 0 for p in blk]
                    ll_loc = n_loc > 0 ? mbp_propose!(store, theta[:, blk], theta_f[:, blk], valid, obs_i) : zeros(2, 0)
                    ll_f = allgather_rows(comm, ll_loc, outer_p, 2)
                    u = rand(outer_p)
                    accepted = [(exp(prior_f[p] - prior[p]) * exp(ll_f[1, p] - log_like[p])) > u[p] for p in 1:outer_p]   # :212
                    mbp_accept!(store, Int64[p - (first(blk) - 1) for p in blk if accepted[p]])       # :214
                    for p in 1:outer_p
                        if accepted[p]
                            mtd_gx[p] = exp(ll_f[2, p]); theta[:, p] = theta_f[:, p]; prior[p] = prior_f[p]; log_like[p] = ll_f[1, p]
                        end
                    end
                    n_acc = count(accepted)
                    k_log[2] += n_acc
                    tj *= alpha^n_acc * 0.999^(outer_p - n_acc)
                end
                bme[2] += log(mlr / Statistics.mean(mtd_gx))
                w .= 1
            else
                bme[2] += log(sum(w .* gx) / sum(w))
            end
        end
    end
    compute_is_mu_covar!(mu, cv, theta, w)
    output = ImportanceSample(mu, cv, theta, w, time_ns() - start_time, -bme)
    comm.rank == 0 && println("- finished in ", print_runtime(output.run_time), " (AR := ", round(100.0 * k_log[2] / k_log[1]; sigdigits = 3), "%)")
    return output
end
