# HmcGPU.jl — Julia binding of libhmcgpu.so (include/hmcgpu.h): the B200 replacement of the Gibbs/FFBS hot loop of Hmc.jl.
#
# Drop-in use from code/run_hmm.jl (replaces `samples = Hmc.estimatemodel(opt)` at line 119):
#
#     include("HmcGPU.jl")
#     samples = HmcGPU.estimatemodel(opt)            # same NamedTuple fields: μ, σ, πb, A, forecasts, obsdates
#     Hmc.saveresults(samples, opt, p; hassignals = false)
#
# and for the noisy-signal blocks (code/run_hmm.jl:133, :151, :174: `samples = Hmc.estimatesignals!(opt)`):
#
#     samples = HmcGPU.estimatesignals!(opt)         # μ, σ, πb, A, forecasts, obsdates, signalvals, signalids
#     Hmc.saveresults(samples, opt, p; hassignals = true)
#
# NOTE: Julia is not installed in the build environment of this repository, so this file has never been executed
# there.  It binds exactly the C ABI that tests/ exercise through Python ctypes (hmc.jl_b200/binding.py); the struct
# layouts below mirror include/hmcgpu.h field by field (checked for the ctypes mirror in tests/test_host.py).
module HmcGPU

using Dates

const LIB = get(ENV, "HMCGPU_LIB", joinpath(@__DIR__, "..", "lib", "libhmcgpu.so"))

const FLAG_REF_Q1 = UInt32(1)
const FLAG_DRAWS = UInt32(2)
const FLAG_SUMMARY = UInt32(4)
const FLAG_SMOOTHED_MEAN = UInt32(8)
const FLAG_FILTERED_MEAN = UInt32(64)
const FLAG_LOGLIK = UInt32(16)
const FLAG_DIAGNOSTICS = UInt32(128)
const FLAG_PREDICTIVE = UInt32(256)
const FLAG_RANKED = UInt32(512)
const FLAG_ONESTEP = UInt32(1024)
const FLAG_LOO = UInt32(2048)

# struct hmcgpu_problem (include/hmcgpu.h)
struct Problem
    y::Ptr{Float64}; y_len::Int64; n_series::Int32; n_windows::Int32
    win_series::Ptr{Int32}; win_start::Ptr{Int32}; win_end::Ptr{Int32}; win_id::Ptr{Int64}
    K::Int32; n_chains::Int32; burnin::Int64; nrun::Int64; seed::UInt64
    xi::Ptr{Float64}; alpha::Ptr{Float64}; nu::Ptr{Float64}; beta0::Ptr{Float64}; beta::Ptr{Float64}
    kappa::Float64; is_signal::Ptr{UInt8}; horizons::Ptr{Int32}; n_h::Int32
    X0::Ptr{Int64}; precision::Int32; flags::UInt32
    win_init_series::Ptr{Int32}; pi_row_back::Int32; is_signal_per_series::Int32
    pred_grid::Ptr{Float64}; n_grid::Int32
end

# struct hmcgpu_result
mutable struct Result
    mu::Ptr{Float64}; sigma2::Ptr{Float64}; A::Ptr{Float64}; pi_end::Ptr{Float64}; forecasts::Ptr{Float64}; loglik::Ptr{Float64}
    summary_mean::Ptr{Float64}; summary_var::Ptr{Float64}; pib_mean::Ptr{Float64}; insample_forecast_mean::Ptr{Float64}; status::Ptr{Int32}
    gpu_ms::Float64; sweep_kernel_ms::Float64; n_launches::Int64; n_sweep_launches::Int64
    h2d_bytes::Int64; d2h_bytes::Int64; state_steps::Int64
    sweep_launch_ms_sum::Float64; sweep_kernel::Int32; n_tasks::Int32
    rhat::Ptr{Float64}; ess::Ptr{Float64}; ess_lag::Ptr{Int32}
end

# struct hmcgpu_predictive (FLAG_PREDICTIVE)
mutable struct Predictive
    cdf::Ptr{Float64}; pit::Ptr{Float64}; log_score::Ptr{Float64}; moments::Ptr{Float64}
end

# struct hmcgpu_ranked (FLAG_RANKED)
mutable struct Ranked
    probs::Ptr{Float64}; n_probs::Int32
    quantiles::Ptr{Float64}; rhat_rank::Ptr{Float64}; ess_bulk::Ptr{Float64}; ess_tail::Ptr{Float64}
end

# struct hmcgpu_onestep (FLAG_ONESTEP)
mutable struct Onestep
    pit::Ptr{Float64}; lpd::Ptr{Float64}; lpd_var::Ptr{Float64}; waic::Ptr{Float64}
end

# struct hmcgpu_loo (FLAG_LOO)
mutable struct Loo
    elpd::Ptr{Float64}; lppd::Ptr{Float64}; pareto_k::Ptr{Float64}; pit::Ptr{Float64}; summary::Ptr{Float64}
end

struct HmcGpuError <: Exception
    code::Int
    msg::String
end

mutable struct Context
    h::Ptr{Cvoid}
    function Context(device::Integer = 0)
        ref = Ref{Ptr{Cvoid}}(C_NULL)
        rc = ccall((:hmcgpu_ctx_create, LIB), Cint, (Cint, Ptr{Ptr{Cvoid}}), device, ref)
        rc == 0 || throw(HmcGpuError(rc, unsafe_string(ccall((:hmcgpu_last_error, LIB), Cstring, (Ptr{Cvoid},), C_NULL))))
        ctx = new(ref[])
        finalizer(c -> (c.h != C_NULL && ccall((:hmcgpu_ctx_destroy, LIB), Cvoid, (Ptr{Cvoid},), c.h); c.h = C_NULL), ctx)
        return ctx
    end
end

lasterror(ctx::Context) = unsafe_string(ccall((:hmcgpu_last_error, LIB), Cstring, (Ptr{Cvoid},), ctx.h))

# Releases the context (stream, device buffers) now instead of whenever the GC runs the finalizer.
function Base.close(ctx::Context)
    ctx.h != C_NULL && ccall((:hmcgpu_ctx_destroy, LIB), Cvoid, (Ptr{Cvoid},), ctx.h)
    ctx.h = C_NULL
    return nothing
end
# Hands the idle device buffers the context keeps for reuse back to the driver (hmcgpu_ctx_trim).
trim(ctx::Context) = ccall((:hmcgpu_ctx_trim, LIB), Cint, (Ptr{Cvoid},), ctx.h)

# One context per device for the whole session: a loop over end dates that calls estimatemodel(opt) must not create a
# context (stream + buffer pool) per call and wait for the GC to release them.
const _contexts = Dict{Int,Context}()
function default_context(device::Integer = 0)
    c = get(_contexts, Int(device), nothing)
    (c === nothing || c.h == C_NULL) && (c = _contexts[Int(device)] = Context(device))
    return c
end

"""
    estimate(ctx, rawdata, win_start, win_end; D, n_chains, burnin, Nrun, seed, horizons, precision)

Many end-date windows in one call (what the SLURM job array of run_hmm.jl does one process at a time).
Returns per-window arrays in the reference's layouts: μ[w] (R×D), σ[w] (R×D), A[w] (R×D×D), πbend[w] (R×D),
forecasts[w] (R×2|H|) with R = n_chains*Nrun (chain-major).  The output buffers are Julia column-major already
(hmcgpu_result), so they are wrapped without a copy.  `onestep = true` adds the one-step-ahead scores of every in-sample
date (hmcgpu_onestep): `onestep_pit[w]`, `lpd[w]` and `lpd_var[w]` (N_w each) and `waic` (4 × nw: lppd, p_waic, elpd_waic, se).
`loo = true` adds PSIS-LOO of every in-sample date (hmcgpu_loo): `loo_elpd[w]`, `loo_lppd[w]`, `pareto_k[w]` and `loo_pit[w]`
(N_w each) and `loo` (6 × nw: elpd_loo, se, p_loo, lppd, max k̂, dates with k̂ above the threshold).
"""
function estimate(ctx::Context, rawdata::VecOrMat{Float64}, win_start::Vector{Int32}, win_end::Vector{Int32};
                  D::Int = 3, n_chains::Int = 1, burnin::Int = 1_000, Nrun::Int = 1_000, seed::Integer = 1234,
                  horizons::Vector{Int32} = Int32[12], precision::Int = 64,
                  win_series::Vector{Int32} = Int32[], win_init_series::Vector{Int32} = Int32[],
                  is_signal::Vector{UInt8} = UInt8[], kappa::Float64 = 1.0, pi_row_back::Int = 0,
                  xi::Vector{Float64} = Float64[], alpha::Vector{Float64} = Float64[], nu::Vector{Float64} = Float64[],
                  pred_grid::Vector{Float64} = Float64[], quantile_probs::Vector{Float64} = Float64[],
                  rank_diagnostics::Bool = false, onestep::Bool = false, loo::Bool = false)
    # rawdata: one series (Vector) or y_len × n_series (Matrix, column = series): exactly the library's column-major layout
    y_len, n_series = size(rawdata, 1), size(rawdata, 2)
    ptr_or_null(v) = isempty(v) ? Ptr{eltype(v)}(C_NULL) : pointer(v)
    nw, nh, R = length(win_start), length(horizons), n_chains * Nrun
    mu = Array{Float64}(undef, R, D, nw); sig = similar(mu); pie = similar(mu)
    A = Array{Float64}(undef, R, D, D, nw)
    fc = Array{Float64}(undef, R, 2nh, nw)
    status = zeros(Int32, n_chains, nw)
    # posterior predictive (non-empty pred_grid): C [w][j][g] row-major = Julia n_grid × n_h × nw
    ng = length(pred_grid)
    pcdf = Array{Float64}(undef, ng, nh, nw); pit = Array{Float64}(undef, nh, nw); pls = similar(pit)
    pmom = Array{Float64}(undef, 3, nh, nw)
    pred = Predictive(pointer(pcdf), pointer(pit), pointer(pls), pointer(pmom))
    # ranked outputs (quantile probabilities or rank_diagnostics): C [w][f][k] row-major = Julia n_probs × F × nw, [w][f] = F × nw
    ranked = !isempty(quantile_probs) || rank_diagnostics
    F, nq = 3D + D * D + 2nh + 1, length(quantile_probs)
    rq = Array{Float64}(undef, nq, F, nw); rrh = Array{Float64}(undef, F, nw); reb = similar(rrh); ret = similar(rrh)
    rk = Ranked(ptr_or_null(quantile_probs), nq, ptr_or_null(rq), pointer(rrh), pointer(reb), pointer(ret))
    # one-step-ahead scores (onestep = true): per date, windows concatenated (split per window below); waic C [w][4] = Julia 4 × nw
    sumT = onestep ? Int(sum(win_end .- win_start .+ 1)) : 0
    opit = Vector{Float64}(undef, sumT); olpd = similar(opit); ovar = similar(opit); owaic = Array{Float64}(undef, 4, onestep ? nw : 0)
    os = Onestep(ptr_or_null(opit), ptr_or_null(olpd), ptr_or_null(ovar), ptr_or_null(owaic))
    # PSIS-LOO (loo = true): per date, windows concatenated; summary C [w][6] = Julia 6 × nw
    sumL = loo ? Int(sum(win_end .- win_start .+ 1)) : 0
    lelpd = Vector{Float64}(undef, sumL); llppd = similar(lelpd); lpk = similar(lelpd); lpit = similar(lelpd)
    lsum = Array{Float64}(undef, 6, loo ? nw : 0)
    lo = Loo(ptr_or_null(lelpd), ptr_or_null(llppd), ptr_or_null(lpk), ptr_or_null(lpit), ptr_or_null(lsum))
    res = Result(pointer(mu), pointer(sig), pointer(A), pointer(pie), nh > 0 ? pointer(fc) : C_NULL, C_NULL,
                 C_NULL, C_NULL, C_NULL, C_NULL, pointer(status), 0.0, 0.0, 0, 0, 0, 0, 0, 0.0, 0, 0,
                 C_NULL, C_NULL, C_NULL)
    rc = GC.@preserve rawdata win_start win_end horizons mu sig A pie fc status win_series win_init_series is_signal xi alpha nu pred_grid pcdf pit pls pmom quantile_probs rq rrh reb ret opit olpd ovar owaic lelpd llppd lpk lpit lsum begin
        prob = Problem(pointer(rawdata), y_len, n_series, nw, ptr_or_null(win_series), pointer(win_start), pointer(win_end), C_NULL,
                       D, n_chains, burnin, Nrun, UInt64(seed), ptr_or_null(xi), ptr_or_null(alpha), ptr_or_null(nu), C_NULL, C_NULL,
                       kappa, ptr_or_null(is_signal), pointer(horizons), nh, C_NULL, precision,
                       FLAG_REF_Q1 | FLAG_DRAWS | (ng > 0 ? FLAG_PREDICTIVE : UInt32(0)) | (ranked ? FLAG_RANKED : UInt32(0)) |
                       (onestep ? FLAG_ONESTEP : UInt32(0)) | (loo ? FLAG_LOO : UInt32(0)),
                       ptr_or_null(win_init_series), pi_row_back, 0, ptr_or_null(pred_grid), ng)
        loo ? ccall((:hmcgpu_estimate_loo, LIB), Cint,
                    (Ptr{Cvoid}, Ref{Problem}, Ref{Result}, Ref{Predictive}, Ref{Ranked}, Ref{Onestep}, Ref{Loo}), ctx.h, prob, res, pred, rk, os, lo) :
        onestep ? ccall((:hmcgpu_estimate_onestep, LIB), Cint,
                        (Ptr{Cvoid}, Ref{Problem}, Ref{Result}, Ref{Predictive}, Ref{Ranked}, Ref{Onestep}), ctx.h, prob, res, pred, rk, os) :
                  ccall((:hmcgpu_estimate_ranked, LIB), Cint, (Ptr{Cvoid}, Ref{Problem}, Ref{Result}, Ref{Predictive}, Ref{Ranked}),
                        ctx.h, prob, res, pred, rk)
    end
    rc < 0 && throw(HmcGpuError(rc, lasterror(ctx)))
    offs = cumsum(vcat(0, Int.(win_end .- win_start .+ 1)))
    per_window(v) = !isempty(v) ? [v[offs[w] + 1:offs[w + 1]] for w in 1:nw] : Vector{Float64}[]
    return (μ = mu, σ = sig, A = A, πbend = pie, forecasts = fc, status = status, events = rc, gpu_ms = res.gpu_ms,
            pred_cdf = pcdf, pit = pit, log_score = pls, pred_moments = pmom,
            quantiles = rq, rhat_rank = rrh, ess_bulk = reb, ess_tail = ret,
            onestep_pit = per_window(opit), lpd = per_window(olpd), lpd_var = per_window(ovar), waic = owaic,
            loo_elpd = per_window(lelpd), loo_lppd = per_window(llppd), pareto_k = per_window(lpk), loo_pit = per_window(lpit), loo = lsum)
end

# The multi-GPU form over caller-built structs (hmcgpu_estimate_multi_ranked): windows sharded over `devices`, every output
# scattered back into the caller's window order.  Returns the event count; throws on an error.
function estimate_multi_ranked(devices::Vector{Cint}, prob::Problem, res::Result, pred::Predictive, rk::Ranked)
    rc = ccall((:hmcgpu_estimate_multi_ranked, LIB), Cint, (Ptr{Cint}, Cint, Ref{Problem}, Ref{Result}, Ref{Predictive}, Ref{Ranked}),
               devices, length(devices), prob, res, pred, rk)
    rc < 0 && throw(HmcGpuError(rc, unsafe_string(ccall((:hmcgpu_last_error, LIB), Cstring, (Ptr{Cvoid},), C_NULL))))
    return rc
end

# The same with the one-step-ahead scores (hmcgpu_estimate_multi_onestep); estimate_multi_ranked is this with os = NULL.
function estimate_multi_onestep(devices::Vector{Cint}, prob::Problem, res::Result, pred::Predictive, rk::Ranked, os::Onestep)
    rc = ccall((:hmcgpu_estimate_multi_onestep, LIB), Cint,
               (Ptr{Cint}, Cint, Ref{Problem}, Ref{Result}, Ref{Predictive}, Ref{Ranked}, Ref{Onestep}),
               devices, length(devices), prob, res, pred, rk, os)
    rc < 0 && throw(HmcGpuError(rc, unsafe_string(ccall((:hmcgpu_last_error, LIB), Cstring, (Ptr{Cvoid},), C_NULL))))
    return rc
end

# The same with the PSIS-LOO outputs (hmcgpu_estimate_multi_loo); estimate_multi_onestep is this with lo = NULL.
function estimate_multi_loo(devices::Vector{Cint}, prob::Problem, res::Result, pred::Predictive, rk::Ranked, os::Onestep, lo::Loo)
    rc = ccall((:hmcgpu_estimate_multi_loo, LIB), Cint,
               (Ptr{Cint}, Cint, Ref{Problem}, Ref{Result}, Ref{Predictive}, Ref{Ranked}, Ref{Onestep}, Ref{Loo}),
               devices, length(devices), prob, res, pred, rk, os, lo)
    rc < 0 && throw(HmcGpuError(rc, unsafe_string(ccall((:hmcgpu_last_error, LIB), Cstring, (Ptr{Cvoid},), C_NULL))))
    return rc
end

# The PSIS-LOO outputs of the last run of a plan (hmcgpu_plan_fetch_loo), computed from the kept draws.  `ctx` is the plan's
# context.
function plan_fetch_loo!(ctx::Context, plan::Ptr{Cvoid}, lo::Loo)
    rc = ccall((:hmcgpu_plan_fetch_loo, LIB), Cint, (Ptr{Cvoid}, Ref{Loo}), plan, lo)
    rc < 0 && throw(HmcGpuError(rc, lasterror(ctx)))
    return lo
end

# The one-step-ahead scores of the last run of a plan (hmcgpu_plan_fetch_onestep).  `ctx` is the plan's context.
function plan_fetch_onestep!(ctx::Context, plan::Ptr{Cvoid}, os::Onestep)
    rc = ccall((:hmcgpu_plan_fetch_onestep, LIB), Cint, (Ptr{Cvoid}, Ref{Onestep}), plan, os)
    rc < 0 && throw(HmcGpuError(rc, lasterror(ctx)))
    return os
end

# The ranked outputs of the last run of a plan (hmcgpu_plan_fetch_ranked), computed from the retained draws; may be called again
# with other rk.probs.  `ctx` is the plan's context (for the error message).
function plan_fetch_ranked!(ctx::Context, plan::Ptr{Cvoid}, rk::Ranked)
    rc = ccall((:hmcgpu_plan_fetch_ranked, LIB), Cint, (Ptr{Cvoid}, Ref{Ranked}), plan, rk)
    rc < 0 && throw(HmcGpuError(rc, lasterror(ctx)))
    return rk
end

# 0/1 flags over rawdata: 1 = the index belongs to opt.signalRange (hmcgpu_problem.is_signal)
signalmask(opt) = (m = zeros(UInt8, length(opt.rawdata)); m[collect(opt.signalRange)] .= 0x01; m)

"""
    estimatemodel(opt; ctx = default_context(0), n_chains = 1, precision = 64)

GPU drop-in for `Hmc.estimatemodel(opt)` (src/Hmc.jl:850-865).  `opt` is an `Hmc.estopt`.  `πb` is returned as an
Nrun×1×D array holding the end-of-window row: `saveresults` reads `samples.πb[:, end, :]` (src/Hmc.jl:744), which works
unchanged; the Nrun×N×D tensor of the reference (3.5 GB per end date in production) is never materialised.
"""
function estimatemodel(opt; ctx::Context = default_context(0), n_chains::Int = 1, precision::Int = 64)
    sr = opt.sampleRange
    # a non-empty signalRange still goes through the signal branches with hp = HyperParams(Y, D), i.e. κ = 1.0 (src/Hmc.jl:853)
    mask = isempty(opt.signalRange) ? UInt8[] : signalmask(opt)
    y = Vector{Float64}(opt.rawdata)
    r = estimate(ctx, y, Int32[first(sr)], Int32[last(sr)]; D = opt.D, n_chains = n_chains,
                 burnin = opt.burnin, Nrun = opt.Nrun, seed = opt.seed, horizons = Int32.(opt.horizons), precision = precision,
                 is_signal = mask, kappa = 1.0)
    R = n_chains * opt.Nrun
    fc = r.forecasts[:, :, 1]
    if last(sr) != opt.endIndex      # :861 scores the forecast from the window END against yobs(endIndex + h)
        for (k, h) in enumerate(opt.horizons)
            fc[:, 2k] = fc[:, 2k - 1] .- (opt.endIndex + h <= length(y) ? y[opt.endIndex + h] : NaN)
        end
    end
    return (μ = r.μ[:, :, 1], σ = r.σ[:, :, 1], πb = reshape(r.πbend[:, :, 1], R, 1, opt.D), A = r.A[:, :, :, 1],
            forecasts = fc, obsdates = fill(opt.dates[opt.endIndex], R))
end

"""
    estimatesignals!(opt; ctx = default_context(0), n_chains = 1, precision = 64)

GPU drop-in for `Hmc.estimatesignals!(opt)` (src/Hmc.jl:868-914).  The `opt.noiseSamples` perturbed copies of the sample
are estimated side by side as independent chains (the reference chains them serially on one state, each with its own
`signalburnin`); priors are `HyperParams(opt)` (α = ν = 2, ξ = mean of the real sample, κ = opt.noise), X0 comes from
`makeParams` on the real data, `πb` is the smoothed row at `opt.endIndex` (:893), forecasts follow :900-906.
Same logic as `estimatesignals` in hmc.jl_b200/api.py, which is the version the GPU tests exercise.
"""
function estimatesignals!(opt; ctx::Context = default_context(0), n_chains::Int = 1, precision::Int = 64)
    if isapprox(opt.σsignal, 0)
        base = estimatemodel(opt; ctx = ctx, n_chains = n_chains, precision = precision)
        opt.σsignal = sum(base.σ) / length(base.σ) * opt.noise
    end
    sr, D, S = opt.sampleRange, opt.D, opt.noiseSamples
    y = Vector{Float64}(opt.rawdata)
    sig = collect(opt.signalRange)
    series = repeat(y, 1, S + 1)                                   # column 1 = real data, 2..S+1 perturbed copies
    series[sig, 2:end] .+= randn(length(sig), S) .* opt.σsignal    # :890
    sigLen = (isempty(sig) ? opt.endIndex : last(sig)) - opt.endIndex
    hs = Int32[max(h - sigLen, 0) for h in opt.horizons]
    xi = fill(sum(y[sr]) / length(sr), D)
    r = estimate(ctx, series, fill(Int32(first(sr)), S), fill(Int32(last(sr)), S); D = D, n_chains = n_chains,
                 burnin = opt.signalburnin, Nrun = opt.signalNrun, seed = opt.seed, horizons = hs, precision = precision,
                 win_series = Int32.(1:S), win_init_series = zeros(Int32, S), is_signal = signalmask(opt), kappa = opt.noise,
                 pi_row_back = last(sr) - opt.endIndex, xi = xi, alpha = fill(2.0, D), nu = fill(2.0, D))
    R = n_chains * opt.signalNrun
    cat2(a) = reduce(vcat, [a[:, :, w] for w in 1:S])
    fc = cat2(r.forecasts)
    for (k, h) in enumerate(opt.horizons)
        yreal = opt.endIndex + h <= length(y) ? y[opt.endIndex + h] : NaN
        if sigLen == h                                              # forecastsignal (:670-681), `noise` = σsignal (:904)
            a = (1 / opt.σsignal) / (1 + 1 / opt.σsignal)
            signal = repeat(series[opt.endIndex + h, 2:end], inner = R)
            fc[:, 2k - 1] = a .* signal .+ (1 - a) .* fc[:, 2k - 1]
            fc[:, 2k] = fc[:, 2k - 1] .- yreal
        elseif sigLen > h
            fc[:, 2k - 1:2k] .= NaN                                 # left unassigned by the reference
        else
            fc[:, 2k] = fc[:, 2k - 1] .- yreal
        end
    end
    save = collect(opt.signalSave)
    return (μ = cat2(r.μ), σ = cat2(r.σ), πb = cat2(r.πbend), A = reduce(vcat, [r.A[:, :, :, w] for w in 1:S]), forecasts = fc,
            obsdates = fill(opt.dates[opt.endIndex], S * R),
            signalvals = repeat(permutedims(series[save, 2:end]), inner = (R, 1)), signalids = repeat(1:S, inner = R))
end

end # module
