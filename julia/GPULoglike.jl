# GPULoglike.jl -- the Julia side of the B200 population step for DifferentialEvolutionMCMC.jl.
#
# STATUS: NOT EXECUTED.  There is no Julia toolchain in the build image or on the GPU box, so this
# file has never been run; every ccall below is exercised through the same ABI by its Python
# ctypes mirror (differentialevolutionmcmc.jl_b200/_ffi.py, handle.py, api.py), which the tests
# drive.  It is written to be `include`d from src/DifferentialEvolutionMCMC.jl after utilities.jl,
# plus `export GPULoglike, GPUPrior` (see INTEGRATION.md).
#
# What it adds to the package:
#   * `GPULoglike(kind; data...)`  -- binds a model to a registered hand-written likelihood kernel
#   * `GPUPrior(specs...)`         -- registered prior specs (one per named parameter)
#   * `GPUDEModel(; prior_loglike, loglike, names, sample_prior)` = `DEModel(loglike::GPULoglike; ...)`:
#     its OWN entry points -- the package's keyword constructor `DEModel(args...; ...)`
#     (src/structs.jl:176-189) is NOT redefined (Julia does not dispatch on keyword types: a method
#     with the same positional signature would replace it and break every CPU model)
#   * `sample(model::DEModel{<:GPULoglike}, de::DE, n_iter)` and the `MCMCThreads()` method:
#     `gpu_sample_init` draws the initial particles exactly as `sample_init` + `init_particle`
#     (src/main.jl:263-271, src/utilities.jl:13-41) but leaves the initial weights to the device
#     (`evaluate_fitness!` would call the plugin object on the host), the state is uploaded, ONE
#     ccall runs all n_iter iterations of step!/pstep! (src/main.jl:84-107) on the device, and the
#     unchanged `bundle_samples` (src/main.jl:222-250) builds the Chains.
# A DEModel whose loglike is any other callable keeps using the package's CPU path; asking for the
# GPU path with a closure throws an ArgumentError -- there is no silent CPU fallback.

const LIBDEMCMC = get(ENV, "LIBDEMCMC_B200", "libdemcmc_b200.so")
const DEMCMC_ABI_VERSION = Int32(8)

const GPU_KINDS = (gaussian = 0, mvnormal = 1, binomial = 2, lnr = 3, lba = 4, hier_normal = 5, rastrigin = 6, mvnormal_full = 7, custom = 8, simulated = 9)
const GPU_PRIORS = (flat = 0, normal = 1, halfcauchy = 2, uniform = 3, beta = 4, normal_ref = 5)

"""
    GPULoglike(kind::Symbol; x = nothing, choice = nothing, rt = nothing, N = nothing, k = nothing,
               sigma = nothing, lba_floor = 1e-10)

`kind ∈ (:gaussian, :mvnormal, :binomial, :lnr, :lba, :hier_normal)`.  `x` is the data vector
(`:gaussian`), the `n_dim × n_obs` matrix handed to `MvNormal` (`:mvnormal`) or the vector of
per-subject vectors / `n_per × n_subj` matrix (`:hier_normal`).

    GPULoglike(:custom, X; source)

A likelihood written as CUDA C++ (`source`, the DEMCMC_CUSTOM contract of include/demcmc_b200.h: `demcmc_obs`, and
optionally `demcmc_particle` / `DEMCMC_NPAR` + `demcmc_prepare`), compiled by the library for sm_100a.  `X` is a vector
(one value per observation), an `n_cols × n_obs` matrix (one column per observation), or `nothing` (no data).

    GPULoglike(:simulated, X; source, n_sim, floor = 1e-10)

A likelihood estimated on the device from `n_sim` simulations per proposal of a simulator written as CUDA C++ (`source`,
the DEMCMC_SIMULATED contract of include/demcmc_b200.h: `demcmc_simulate(par, rng, y)` with `demcmc_uniform` /
`demcmc_normal`, and optionally `DEMCMC_NPAR` + `demcmc_prepare`): a Gaussian kernel density per label, Silverman's
bandwidth, floored at `floor`.  `X` is a vector of values, or a `2 × n_obs` matrix of (label 1..8, value) columns.  Only
proposals are simulated: a particle keeps the estimate it was accepted with (pseudo-marginal).
"""
struct GPULoglike{D}
    kind::Symbol
    data::D
    sigma::Union{Nothing, Vector{Float64}}
    lba_floor::Float64
    cov::Matrix{Float64}   # :mvnormal_full: the known covariance Σ of MvNormal(μ, σ²Σ); empty otherwise
    source::String         # :custom / :simulated: the CUDA C++ source of the likelihood / simulator; empty otherwise
    n_sim::Int32           # :simulated: simulations per proposal; 0 otherwise
    sim_floor::Float64     # :simulated: density floor
end

function GPULoglike(kind::Symbol; x = nothing, choice = nothing, rt = nothing, N = nothing, k = nothing,
    sigma = nothing, lba_floor = 1e-10, cov = zeros(0, 0))
    haskey(GPU_KINDS, kind) || throw(ArgumentError("no registered kernel for :$kind; registered: $(keys(GPU_KINDS))"))
    data = if kind == :binomial
        (x = Float64[N, k], choice = nothing)
    elseif kind in (:lnr, :lba)
        (x = Vector{Float64}(rt), choice = Vector{Int32}(choice))
    elseif kind == :hier_normal && x isa AbstractVector{<:AbstractVector}
        (x = Matrix{Float64}(reduce(hcat, x)), choice = nothing)   # n_per × n_subj == C [n_subj][n_per]
    else
        (x = Array{Float64}(x), choice = nothing)
    end
    kind == :mvnormal_full && size(cov) != (size(data.x, 1), size(data.x, 1)) && throw(ArgumentError(":mvnormal_full needs cov, n_dim × n_dim"))
    return GPULoglike(kind, data, sigma === nothing ? nothing : Vector{Float64}(sigma), Float64(lba_floor), Matrix{Float64}(cov), "", Int32(0), 1e-10)
end

# the source is compiled when the model is bound (demcmc_set_model caches the cubin per source text); a source that
# does not compile raises there, with the compiler log as the library's error message.  :simulated data and arguments are
# checked again by demcmc_set_model.
function GPULoglike(kind::Symbol, X; source::AbstractString, n_sim::Integer = 0, floor::Real = 1e-10)
    kind in (:custom, :simulated) || throw(ArgumentError("GPULoglike(kind, X; source) is the :custom / :simulated form"))
    isempty(source) && throw(ArgumentError(":$kind needs the CUDA source of " * (kind == :custom ? "demcmc_obs" : "demcmc_simulate")))
    if kind == :custom
        x = X === nothing ? zeros(0, 0) : X isa AbstractVector ? Matrix{Float64}(reshape(X, 1, :)) : Matrix{Float64}(X)
        (X !== nothing && size(x, 1) == 0) && throw(ArgumentError(":custom data need at least one value per observation"))
        return GPULoglike(kind, (x = x, choice = nothing), nothing, 1e-10, zeros(0, 0), String(source), Int32(0), 1e-10)
    end
    16 <= n_sim <= 16384 || throw(ArgumentError(":simulated needs 16 <= n_sim <= 16384, got $n_sim"))
    floor > 0 || throw(ArgumentError(":simulated needs floor > 0, got $floor"))
    x = X isa AbstractVector ? Matrix{Float64}(reshape(X, 1, :)) : Matrix{Float64}(X)
    size(x, 1) in (1, 2) || throw(ArgumentError(":simulated data are values or (label, value) columns"))
    return GPULoglike(kind, (x = x, choice = nothing), nothing, 1e-10, zeros(0, 0), String(source), Int32(n_sim), Float64(floor))
end

# the device evaluates it; calling it on the host is an error, never a fallback
(::GPULoglike)(args...; kwargs...) =
    throw(ArgumentError("GPULoglike is evaluated by libdemcmc_b200 on the device; it is not a host function"))

"Registered prior specs: `(:normal, μ, σ)`, `(:halfcauchy, loc, scale)` = truncated(Cauchy(loc,scale),0,Inf), `(:uniform, a, b)`, `(:beta, a, b)`, `(:flat,)`, `(:normal_ref, mean, :name_of_sd_parameter)`."
struct GPUPrior
    specs::Vector{Tuple}
end
GPUPrior(specs::Tuple...) = GPUPrior(collect(Tuple, specs))

# The package's keyword constructor DEModel(args...; prior_loglike, loglike, names, sample_prior, data, kwargs...)
# (src/structs.jl:176-189) wraps loglike / prior_loglike in closures, which would hide the plugin object -- and it
# must stay as it is for every CPU model.  A GPU model therefore has its OWN constructors, which store the plugin
# unwrapped through the positional inner constructor DEModel(prior_loglike, loglike, sample_prior, names)
# (src/structs.jl:169-174):
#   GPUDEModel(; prior_loglike = GPUPrior(...), loglike = GPULoglike(...), names, sample_prior)
#   DEModel(GPULoglike(...); prior_loglike = GPUPrior(...), names, sample_prior)     # one POSITIONAL plugin argument
# (the second is a distinct, more specific method than DEModel(args...; ...): it does not replace it).
# prior_loglike may be `nothing` for optimize with evaluate_fun! (src/utilities.jl:113-120 never calls it).
function GPUDEModel(; prior_loglike::Union{GPUPrior, Nothing} = nothing, loglike::GPULoglike, names, sample_prior)
    return DEModel(prior_loglike, loglike, sample_prior, names)
end
function DEModel(loglike::GPULoglike; prior_loglike::Union{GPUPrior, Nothing} = nothing, names, sample_prior)
    return GPUDEModel(; prior_loglike, loglike, names, sample_prior)
end

# sample_init (src/main.jl:263-271) + init_particle (src/utilities.jl:13-22) for a GPU model: the same
# de.samples array (initialize_samples, src/utilities.jl:29-41, unchanged: it only calls model.sample_prior()), the
# same sample_prior() call per particle in id order, the same zeroed accept / lp vectors -- but NOT
# de.evaluate_fitness!(de, model, p): that would call the GPULoglike / GPUPrior objects on the host.  The initial
# weights are computed by demcmc_set_state on the device.
function gpu_sample_init(model::DEModel, de::DE, n_iter)
    de.samples = initialize_samples(de, model, n_iter)
    N = n_iter + de.n_initial
    id = 0
    groups = [[begin
                   id += 1
                   Θ = de.n_initial > 0 ? de.samples[1, :, id] : model.sample_prior()
                   p = Particle(; Θ, id)
                   p.accept = fill(false, N)
                   p.lp = fill(0.0, N)
                   p
               end for _ = 1:(de.Np)] for _ = 1:(de.n_groups)]
    return groups
end

# ---- C structs (include/demcmc_b200.h) -----------------------------------------------------------
struct CPrior
    kind::Int32
    ref::Int32
    a::Float64
    b::Float64
end

struct CModel
    kind::Int32
    d::Int32
    n_obs::Int64
    n_dim::Int32
    n_per::Int32
    x::Ptr{Float64}
    choice::Ptr{Int32}
    sigma::Ptr{Float64}
    lba_floor::Float64
    prior::Ptr{CPrior}
    data_on_device::Int32
    n_cols::Int32          # :custom: values per observation (rows of the n_cols × n_obs data matrix)
    cov::Ptr{Float64}      # :mvnormal_full: the known covariance, n_dim × n_dim
    center::Ptr{Float64}   # C_NULL: centre the data on their column means (the product default)
    source::Ptr{UInt8}     # :custom / :simulated: NUL-terminated CUDA source (a Julia String's pointer), else C_NULL
    n_sim::Int32           # :simulated: simulations per proposal
    sim_floor::Float64     # :simulated: density floor
end

struct CConfig
    abi_version::Int32
    n_groups::Int32
    Np::Int32
    d::Int32
    burnin::Int32
    n_initial::Int32
    alpha::Float64
    beta::Float64
    eps::Float64
    sigma::Float64
    kappa::Float64
    theta_snooker::Float64
    proposal::Int32
    n_blocks::Int32
    blocks::Ptr{UInt8}
    lo::Ptr{Float64}
    hi::Ptr{Float64}
    seed::UInt64
    device::Int32
    group_begin::Int32
    group_count::Int32
    donors::Int32          # 0 = sample (current group), 1 = resample (history, DE-MCz)
    trace::Int32
    store_every::Int32
    update::Int32          # 0 mh_update!, 1 maximize!, 2 minimize!
    fitness::Int32         # 0 compute_posterior!, 1 evaluate_fun!
    n_devices::Int32       # > 1: ONE handle over several GPUs of the box, driven from this one Julia process
    devices::Ptr{Int32}    # [n_devices] CUDA ordinals
end

function demcmc_check(rc)
    rc == 0 && return nothing
    msg = unsafe_string(ccall((:demcmc_last_error, LIBDEMCMC), Cstring, ()))
    error("libdemcmc_b200 error $rc: $msg")
end

# flattening in `names` order, column-major inside array parameters (get_names, src/utilities.jl:131-149)
flatten_theta(Θ) = Float64[x for θ in Θ for x in (θ isa AbstractArray ? vec(θ) : (θ,))]
n_elems(θ) = θ isa AbstractArray ? length(θ) : 1

function expand_bounds(bounds, Θ)
    lo, hi = Float64[], Float64[]
    for (i, θ) in enumerate(Θ)
        b = i <= length(bounds) ? bounds[i] : (-Inf, Inf)      # zip truncation, src/utilities.jl:74
        append!(lo, fill(Float64(b[1]), n_elems(θ)))
        append!(hi, fill(Float64(b[2]), n_elems(θ)))
    end
    return lo, hi
end

function expand_block(block, Θ)
    out = UInt8[]
    for (b, θ) in zip(block, Θ)
        append!(out, b isa AbstractArray ? UInt8.(vec(b)) : fill(UInt8(b), n_elems(θ)))
    end
    return out
end

function prior_table(model, Θ)
    starts = Dict{Symbol, Int}()
    pos = 0
    for (n, θ) in zip(model.names, Θ)
        starts[Symbol(n)] = pos
        pos += n_elems(θ)
    end
    table = CPrior[]
    model.prior_loglike === nothing && return fill(CPrior(GPU_PRIORS[:flat], 0, 0.0, 0.0), pos)   # evaluate_fun! never calls it
    for (spec, θ) in zip(model.prior_loglike.specs, Θ)
        kind = GPU_PRIORS[spec[1]]
        a = length(spec) > 1 ? Float64(spec[2]) : 0.0
        if spec[1] == :normal_ref
            append!(table, fill(CPrior(kind, starts[Symbol(spec[3])], a, 0.0), n_elems(θ)))
        else
            b = length(spec) > 2 ? Float64(spec[3]) : 0.0
            append!(table, fill(CPrior(kind, 0, a, b), n_elems(θ)))
        end
    end
    return table
end

proposal_id(de) = de.generate_proposal === random_gamma ? 0 : de.generate_proposal === fixed_gamma ? 1 :
                  de.generate_proposal === variable_gamma ? 2 :
                  throw(ArgumentError("generate_proposal must be random_gamma, fixed_gamma or variable_gamma on the B200 path"))

# ---- the sampler ---------------------------------------------------------------------------------
# `devices = [0, 1, ..., 7]`: the groups shard over several GPUs of the box from THIS process (demcmc_config.n_devices:
# one host thread of the library per GPU, migration over NVLink through peer-mapped mailboxes) -- what replaces the
# ThreadsX.map over groups of p_update! (src/main.jl:135-148); no MPI, no second process.  `store_every = k` keeps
# iterations k, 2k, ... only (the Chains then hold (n_iter - burnin) ÷ k draws).
function sample(model::DEModel{<:GPULoglike}, de::DE, n_iter::Int; progress = false, device = 0, devices = Int32[], store_every = 1, seed = rand(UInt64), kwargs...)
    return _sample_gpu(model, de, n_iter; device, devices, store_every, seed)
end
function sample(model::DEModel{<:GPULoglike}, de::DE, ::MCMCThreads, n_iter::Int; progress = false, device = 0, devices = Int32[], store_every = 1, seed = rand(UInt64), kwargs...)
    return _sample_gpu(model, de, n_iter; device, devices, store_every, seed)    # every group is always updated concurrently on the device(s)
end

# demcmc_model's n_dim, n_per, n_obs, n_cols of a GPULoglike with d flattened parameters
function model_geometry(ll::GPULoglike, d)
    x = ll.data.x
    n_dim, n_per, n_obs, n_cols = 0, 0, length(x), 0
    if ll.kind == :custom || ll.kind == :simulated
        n_cols, n_obs = size(x)
    elseif ll.kind == :mvnormal || ll.kind == :mvnormal_full
        n_dim, n_obs = size(x)
    elseif ll.kind == :hier_normal
        n_per, n_dim = size(x); n_obs = n_dim * n_per
    elseif ll.kind == :lnr
        n_dim = d - 1
    elseif ll.kind == :lba
        n_dim = d - 3
    elseif ll.kind == :binomial
        n_obs = 1
    end
    return n_dim, n_per, n_obs, n_cols
end

function _sample_gpu(model, de, n_iter; device, seed, devices = Int32[], store_every = 1, return_particles = false, temperatures = nothing,
                     evidence = nothing)
    store_every == 1 || return_particles === false || throw(ArgumentError("optimize keeps every row"))
    store_every == 1 || return _sample_gpu_thinned(model, de, n_iter; device, devices, store_every, seed)
    devs = Vector{Int32}(devices)
    model.prior_loglike isa GPUPrior || de.evaluate_fitness! === evaluate_fun! ||
        throw(ArgumentError("prior_loglike must be a GPUPrior: a Julia closure would need a host round trip per particle"))
    update = de.update_particle! === mh_update! ? Int32(0) : de.update_particle! === maximize! ? Int32(1) :
             de.update_particle! === minimize! ? Int32(2) : throw(ArgumentError("update_particle! must be mh_update!, maximize! or minimize!"))
    fitness = de.evaluate_fitness! === compute_posterior! ? Int32(0) : de.evaluate_fitness! === evaluate_fun! ? Int32(1) :
              throw(ArgumentError("evaluate_fitness! must be compute_posterior! or evaluate_fun!"))
    de.sample === sample || de.sample === resample ||
        throw(ArgumentError("de.sample must be `sample` or `resample`: a custom donor function cannot run on the device"))
    donors = de.sample === resample ? Int32(1) : Int32(0)
    ll = model.loglike
    # initial Θ and ids drawn exactly as sample_init does (src/main.jl:263-271), weights left to the device
    groups = gpu_sample_init(model, de, n_iter)
    particles = vcat(groups...)
    Θ1 = particles[1].Θ
    d = sum(n_elems, Θ1)
    P = length(particles)
    theta0 = reduce(hcat, (flatten_theta(p.Θ) for p in particles))          # d × P == C [P][d]
    lo, hi = expand_bounds(de.bounds, Θ1)
    # blocking_on(de) is evaluated every iteration with de.iter = iter + n_initial (src/main.jl:34,137,162)
    iter_keep = de.iter
    block_on = UInt8[(de.iter = it + de.n_initial; de.blocking_on(de) ? 1 : 0) for it = 1:n_iter]
    de.iter = iter_keep
    blocks = any(!iszero, block_on) ? reduce(vcat, (expand_block(b, Θ1) for b in de.blocks)) : UInt8[]
    n_blocks = any(!iszero, block_on) ? length(de.blocks) : 0
    priors = prior_table(model, Θ1)
    x = ll.data.x
    choice = ll.data.choice
    n_dim, n_per, n_obs, n_cols = model_geometry(ll, d)
    covm = ll.cov
    src = ll.source
    h = Ref{Ptr{Cvoid}}(C_NULL)
    n_rows = n_iter + de.n_initial
    samples = zeros(Float64, n_rows, d, P)          # Julia order == the library's output order
    accept = zeros(UInt8, n_rows, P)
    lp = zeros(Float64, n_rows, P)
    final_ids = zeros(Int32, P)
    final_theta = zeros(Float64, d, P)               # d × P == C [P][d]
    final_weight = zeros(Float64, P)
    # initialize_samples (src/utilities.jl:29-41) already filled rows 1:n_initial of de.samples with
    # prior draws; the library wants them as [n_initial][P][d]
    init_rows = de.n_initial > 0 ?
        Float64[flatten_theta(de.samples[i, :, p])[k] for k = 1:d, p = 1:P, i = 1:(de.n_initial)] : Float64[]
    sig = ll.sigma === nothing ? Float64[] : ll.sigma
    GC.@preserve theta0 lo hi blocks priors x choice sig covm src samples accept lp final_ids final_theta final_weight init_rows devs begin
        cfg = CConfig(DEMCMC_ABI_VERSION, de.n_groups, de.Np, d, de.burnin, de.n_initial, de.α, de.β, de.ϵ, de.σ, de.κ,
            de.θsnooker, proposal_id(de), n_blocks, isempty(blocks) ? C_NULL : pointer(blocks), pointer(lo), pointer(hi),
            seed, device, 0, 0, donors, 0, 1, update, fitness, length(devs), isempty(devs) ? C_NULL : pointer(devs))
        demcmc_check(ccall((:demcmc_create, LIBDEMCMC), Cint, (Ref{CConfig}, Ref{Ptr{Cvoid}}), cfg, h))
        try
            m = CModel(GPU_KINDS[ll.kind], d, n_obs, n_dim, n_per, pointer(x), choice === nothing ? C_NULL : pointer(choice),
                isempty(sig) ? C_NULL : pointer(sig), ll.lba_floor, pointer(priors), 0, n_cols, isempty(covm) ? C_NULL : pointer(covm), C_NULL,
                isempty(src) ? C_NULL : pointer(src), ll.n_sim, ll.sim_floor)
            demcmc_check(ccall((:demcmc_set_model, LIBDEMCMC), Cint, (Ptr{Cvoid}, Ref{CModel}), h[], m))
            if n_blocks > 0 && !all(!iszero, block_on)         # block updating in some iterations only
                GC.@preserve block_on demcmc_check(ccall((:demcmc_set_blocking_schedule, LIBDEMCMC), Cint, (Ptr{Cvoid}, Ptr{UInt8}, Int64), h[], block_on, length(block_on)))
            end
            if de.n_initial > 0
                demcmc_check(ccall((:demcmc_set_history, LIBDEMCMC), Cint, (Ptr{Cvoid}, Ptr{Float64}), h[], init_rows))
            end
            if temperatures !== nothing                        # power_posterior: one temperature per group, before the weights
                set_temperatures!(h[], temperatures)
            end
            # init_particle (src/utilities.jl:13-22) already started every particle from samples[1, :, id]
            # when n_initial > 0, so theta0 is right in both cases
            demcmc_check(ccall((:demcmc_set_state, LIBDEMCMC), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Int32}), h[], theta0, C_NULL))
            demcmc_check(ccall((:demcmc_run, LIBDEMCMC), Cint, (Ptr{Cvoid}, Int64), h[], n_iter))
            if evidence !== nothing                            # every row after burn-in, as bundle_samples drops it
                row0 = max(de.discard_burnin ? de.burnin : 0, de.n_initial)
                evidence[] = handle_power_posterior(h[], row0, n_rows - row0, de.n_groups)
            end
            demcmc_check(ccall((:demcmc_get_samples, LIBDEMCMC), Cint, (Ptr{Cvoid}, Ptr{Float64}, Int64), h[], samples, n_rows))
            demcmc_check(ccall((:demcmc_get_accept, LIBDEMCMC), Cint, (Ptr{Cvoid}, Ptr{UInt8}, Int64), h[], accept, n_rows))
            demcmc_check(ccall((:demcmc_get_lp, LIBDEMCMC), Cint, (Ptr{Cvoid}, Ptr{Float64}, Int64), h[], lp, n_rows))
            demcmc_check(ccall((:demcmc_get_state, LIBDEMCMC), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}), h[], final_theta, final_weight, final_ids))
        finally
            ccall((:demcmc_destroy, LIBDEMCMC), Cint, (Ptr{Cvoid},), h[])
        end
    end
    # rebuild what bundle_samples reads: de.samples (nested per named parameter) and, at final
    # position c, the accept/lp history of the particle that ended there (src/main.jl:232-241)
    de.iter = n_iter + de.n_initial
    de.samples = nest_samples(samples, Θ1)
    for (c, p) in enumerate(particles)
        id = final_ids[c] + 1
        p.accept = Bool.(accept[:, id])
        p.lp = lp[:, id]
    end
    if return_particles                              # optimize: vcat(groups...) in final position order
        for (c, p) in enumerate(particles)
            k = 0
            p.Θ = as_union([begin n = n_elems(θ); v = θ isa AbstractArray ? reshape(final_theta[(k + 1):(k + n), c], size(θ)) : final_theta[k + 1, c]; k += n; v end for θ in Θ1])
            p.weight = final_weight[c]
            p.id = final_ids[c] + 1
        end
        return nothing, particles
    end
    groups = [particles[((g - 1) * de.Np + 1):(g * de.Np)] for g = 1:(de.n_groups)]
    return bundle_samples(model, de, groups, n_iter)
end

# Thinned run (store_every = k > 1): de.samples would have holes, so the Chains are built from the device-side
# bundle_samples (demcmc_get_chains) of the kept rows instead of from de.samples.
function _sample_gpu_thinned(model, de, n_iter; device, devices, store_every, seed)
    groups = gpu_sample_init(model, de, 0)               # initial draws only; no n_iter-long host arrays
    particles = vcat(groups...)
    Θ1 = particles[1].Θ
    d = sum(n_elems, Θ1); P = length(particles)
    theta0 = reduce(hcat, (flatten_theta(p.Θ) for p in particles))
    lo, hi = expand_bounds(de.bounds, Θ1)
    priors = prior_table(model, Θ1)
    ll = model.loglike
    ll.kind in (:gaussian, :mvnormal, :hier_normal) || throw(ArgumentError("thinned runs are wired for the matrix / vector data kinds in this wrapper"))
    de.n_initial == 0 || throw(ArgumentError("store_every > 1 with n_initial > 0: use the full-history path"))
    de.blocking_on(de) && throw(ArgumentError("store_every > 1 with blocks: use the full-history path"))
    x = ll.data.x
    n_dim, n_per, n_obs = ll.kind == :mvnormal ? (size(x, 1), 0, size(x, 2)) : ll.kind == :hier_normal ? (size(x, 2), size(x, 1), length(x)) : (0, 0, length(x))
    devs = Vector{Int32}(devices)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    local v
    GC.@preserve theta0 lo hi priors x devs begin
        cfg = CConfig(DEMCMC_ABI_VERSION, de.n_groups, de.Np, d, de.burnin, 0, de.α, de.β, de.ϵ, de.σ, de.κ, de.θsnooker, proposal_id(de), 0, C_NULL,
            pointer(lo), pointer(hi), seed, device, 0, 0, 0, 0, store_every, 0, 0, length(devs), isempty(devs) ? C_NULL : pointer(devs))
        demcmc_check(ccall((:demcmc_create, LIBDEMCMC), Cint, (Ref{CConfig}, Ref{Ptr{Cvoid}}), cfg, h))
        try
            m = CModel(GPU_KINDS[ll.kind], d, n_obs, n_dim, n_per, pointer(x), C_NULL, C_NULL, ll.lba_floor, pointer(priors), 0, 0, C_NULL, C_NULL, C_NULL, Int32(0), 1e-10)
            demcmc_check(ccall((:demcmc_set_model, LIBDEMCMC), Cint, (Ptr{Cvoid}, Ref{CModel}), h[], m))
            demcmc_check(ccall((:demcmc_set_state, LIBDEMCMC), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Int32}), h[], theta0, C_NULL))
            demcmc_check(ccall((:demcmc_run, LIBDEMCMC), Cint, (Ptr{Cvoid}, Int64), h[], n_iter))
            offset = de.discard_burnin ? de.burnin ÷ store_every : 0
            Ns = n_iter ÷ store_every - offset
            v = zeros(Float64, Ns, d + 2, P)
            GC.@preserve v demcmc_check(ccall((:demcmc_get_chains, LIBDEMCMC), Cint, (Ptr{Cvoid}, Int64, Int64, Ptr{Float64}), h[], offset, Ns, v))
        finally
            ccall((:demcmc_destroy, LIBDEMCMC), Cint, (Ptr{Cvoid},), h[])
        end
    end
    de.iter = n_iter
    return Chains(v, get_names(model, particles[1]), (parameters = [model.names...], internals = ["acceptance", "lp"]))
end

# Faster exit when only the Chains are wanted: bundle_samples (src/main.jl:222-250) runs on the device
# and one download returns its Array{Float64,3}(Ns, d + 2, P) in Julia order, ready for
# `Chains(v, all_names, (parameters = [model.names...], internals = ["acceptance", "lp"]))`.
function device_bundle(h, de, n_iter, d, P)
    Ns = de.discard_burnin ? n_iter - de.burnin : n_iter
    offset = de.discard_burnin ? de.burnin : 0
    v = zeros(Float64, Ns, d + 2, P)
    GC.@preserve v demcmc_check(ccall((:demcmc_get_chains, LIBDEMCMC), Cint, (Ptr{Cvoid}, Int64, Int64, Ptr{Float64}), h, offset, Ns, v))
    return v
end

# Checkpoint / resume: `state = device_state(h)` after `n_done` iterations; later, on a fresh handle,
# `resume!(h2, state, n_done)` and the chain continues exactly (same Philox counters, burn-in switch and
# migration schedule) -- the reference itself has no such facility (its RNG is the task-local one).
function device_state(h, P, d)
    θ = zeros(Float64, d, P); w = zeros(Float64, P); ids = zeros(Int32, P)
    GC.@preserve θ w ids demcmc_check(ccall((:demcmc_get_state, LIBDEMCMC), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}), h, θ, w, ids))
    return (θ = θ, w = w, ids = ids)
end
function resume!(h, state, n_done)
    GC.@preserve state begin
        demcmc_check(ccall((:demcmc_set_state, LIBDEMCMC), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Int32}), h, state.θ, state.ids))
        demcmc_check(ccall((:demcmc_set_weights, LIBDEMCMC), Cint, (Ptr{Cvoid}, Ptr{Float64}), h, state.w))
    end
    demcmc_check(ccall((:demcmc_set_iteration, LIBDEMCMC), Cint, (Ptr{Cvoid}, Int64), h, n_done))
end

# Pooled posterior mean / variance of the flattened parameters over rows offset+1 .. offset+Ns of
# de.samples, computed on the device: what `describe(chains)` reports as mean and std, without the
# download of the draws (configs[4] would hand 423 GB to the host).
function device_moments(h, offset, Ns, d)
    count = Ref{Int64}(0)
    mean = zeros(Float64, d); m2 = zeros(Float64, d)
    GC.@preserve mean m2 demcmc_check(ccall((:demcmc_get_moments, LIBDEMCMC), Cint,
        (Ptr{Cvoid}, Int64, Int64, Ref{Int64}, Ptr{Float64}, Ptr{Float64}), h, offset, Ns, count, mean, m2))
    return count[], mean, m2 ./ max(count[] - 1, 1)
end

# [n_iter, d, P] flat -> the reference's Array{T,3}(n_iter, n_named, P) whose elements may be arrays
function nest_samples(flat, Θ1)
    n_iter, _, P = size(flat)
    out = Array{eltype(Θ1), 3}(undef, n_iter, length(Θ1), P)
    for c = 1:P, s = 1:n_iter
        k = 0
        for (ni, θ) in enumerate(Θ1)
            n = n_elems(θ)
            out[s, ni, c] = θ isa AbstractArray ? reshape(flat[s, (k + 1):(k + n), c], size(θ)) : flat[s, k + 1, c]
            k += n
        end
    end
    return out
end


# optimize(model, de, n_iter) (src/optimize.jl:17-66) for a GPULoglike model: the same device loop with
# de.update_particle! = maximize!/minimize! and de.evaluate_fitness! = evaluate_fun! (both travel in
# demcmc_config.update / .fitness).  _sample_gpu already rebuilt de.samples; the particles come back
# from the final rows of it plus demcmc_get_state, so get_optimal(de, model, particles)
# (src/utilities.jl:258-266) works unchanged.
function optimize(model::DEModel{<:GPULoglike}, de::DE, n_iter::Int; progress = false, device = 0, seed = rand(UInt64), kwargs...)
    _, particles = _sample_gpu(model, de, n_iter; device, seed, return_particles = true)
    return particles
end
optimize(model::DEModel{<:GPULoglike}, de::DE, ::MCMCThreads, n_iter::Int; kwargs...) = optimize(model, de, n_iter; kwargs...)

# ---- model comparison ------------------------------------------------------------------------------------------------
# log p(y_i | θ) of every observation under every draw, and PSIS-LOO / WAIC, on the device (demcmc_eval_pointwise /
# demcmc_loo, include/demcmc_b200.h).  Both leave the priors out and need no run: the handle is bound to the likelihood
# alone.  `f(h, theta, n, n_obs)` runs on that handle with the draws of `chains` as theta[d][n], chain by chain.
function _with_likelihood(f, model::DEModel{<:GPULoglike}, chains; device = 0)
    v = Array(chains.value)                                  # Ns × (d + 2) × n_chains; acceptance and lp last
    d = size(v, 2) - 2
    theta = reshape(permutedims(v[:, 1:d, :], (2, 1, 3)), d, :)
    ll = model.loglike
    n_dim, n_per, n_obs, n_cols = model_geometry(ll, d)
    x, choice, covm, src = ll.data.x, ll.data.choice, ll.cov, ll.source
    sig = ll.sigma === nothing ? Float64[] : ll.sigma
    lo, hi = fill(-Inf, d), fill(Inf, d)
    priors = [CPrior(Int32(GPU_PRIORS.flat), Int32(0), 0.0, 0.0) for _ in 1:d]
    h = Ref{Ptr{Cvoid}}(C_NULL)
    GC.@preserve theta x choice sig covm src lo hi priors begin
        cfg = CConfig(DEMCMC_ABI_VERSION, 1, 3, d, 0, 0, 0.0, 0.0, 0.001, 0.05, 1.0, 0.0, Int32(0), 0, C_NULL, pointer(lo), pointer(hi),
            UInt64(0), device, 0, 0, 0, 0, 1, 0, 0, 0, C_NULL)
        demcmc_check(ccall((:demcmc_create, LIBDEMCMC), Cint, (Ref{CConfig}, Ref{Ptr{Cvoid}}), cfg, h))
        try
            m = CModel(GPU_KINDS[ll.kind], d, n_obs, n_dim, n_per, pointer(x), choice === nothing ? C_NULL : pointer(choice),
                isempty(sig) ? C_NULL : pointer(sig), ll.lba_floor, pointer(priors), 0, n_cols, isempty(covm) ? C_NULL : pointer(covm), C_NULL,
                isempty(src) ? C_NULL : pointer(src), ll.n_sim, ll.sim_floor)
            demcmc_check(ccall((:demcmc_set_model, LIBDEMCMC), Cint, (Ptr{Cvoid}, Ref{CModel}), h[], m))
            return f(h[], theta, size(theta, 2), n_obs), size(v, 1), size(v, 3)
        finally
            ccall((:demcmc_destroy, LIBDEMCMC), Cint, (Ptr{Cvoid},), h[])
        end
    end
end

# n_obs × n_steps × n_chains, the [data, step, chain] array ParetoSmooth.psis_loo takes:
#   psis_loo(pointwise_loglikelihoods(model, chains))
function pointwise_loglikelihoods(model::DEModel{<:GPULoglike}, chains; device = 0)
    out, Ns, nc = _with_likelihood(model, chains; device) do h, theta, n, n_obs
        ll = zeros(Float64, n_obs, n)                         # Julia n_obs × n == C out[n][n_obs]
        GC.@preserve ll demcmc_check(ccall((:demcmc_eval_pointwise, LIBDEMCMC), Cint,
            (Ptr{Cvoid}, Ptr{Float64}, Int64, Int64, Int64, Ptr{Float64}), h, theta, n, 0, n_obs, ll))
        ll
    end
    return reshape(out, :, Ns, nc)
end

# PSIS-LOO and WAIC with Pareto smoothing on the device (at most DEMCMC_LOO_MAX_DRAWS = 16384 draws: thin longer chains)
function loo(model::DEModel{<:GPULoglike}, chains; device = 0)
    (elpd_i, k, lppd_i, pw_i), _, _ = _with_likelihood(model, chains; device) do h, theta, n, n_obs
        o = ntuple(_ -> zeros(Float64, n_obs), 4)
        GC.@preserve o demcmc_check(ccall((:demcmc_loo, LIBDEMCMC), Cint,
            (Ptr{Cvoid}, Ptr{Float64}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}), h, theta, n, o[1], o[2], o[3], o[4]))
        o
    end
    N = length(elpd_i)
    waic_i = lppd_i .- pw_i
    se(a) = sqrt(N * sum(abs2, a .- sum(a) / N) / N)
    return (elpd_loo = sum(elpd_i), se_elpd_loo = se(elpd_i), p_loo = sum(lppd_i) - sum(elpd_i), elpd_waic = sum(waic_i),
            se_elpd_waic = se(waic_i), p_waic = sum(pw_i), n_bad_k = count(>(0.7), k), elpd_loo_i = elpd_i, pareto_k = k,
            lppd_i = lppd_i, p_waic_i = pw_i)
end

# ---- power posteriors: the marginal likelihood log p(y | M) (include/demcmc_b200.h: demcmc_power_posterior) ----------------
struct CEvidence
    n_rungs::Int32
    log_z_ti::Float64
    log_z_ti2::Float64
    log_z_ss::Float64
    se_ti::Float64
    se_ss::Float64
end

# t[g] in [0, 1] for every group of the job: after demcmc_set_model, before demcmc_set_state
set_temperatures!(h::Ptr{Cvoid}, t::AbstractVector{<:Real}) = (tt = Vector{Float64}(t);
    GC.@preserve tt demcmc_check(ccall((:demcmc_set_temperatures, LIBDEMCMC), Cint, (Ptr{Cvoid}, Ptr{Float64}, Int32), h, tt, length(tt))))

# the stored untempered log-likelihoods, n_rows × P like Particle.lp (the n_initial prior rows are NaN)
function get_loglike(h::Ptr{Cvoid}, n_rows, P)
    out = zeros(Float64, n_rows, P)
    GC.@preserve out demcmc_check(ccall((:demcmc_get_loglike, LIBDEMCMC), Cint, (Ptr{Cvoid}, Ptr{Float64}, Int64), h, out, n_rows))
    return out
end

function handle_power_posterior(h::Ptr{Cvoid}, row0, n_rows, cap)
    ev = Ref{CEvidence}()
    a = ntuple(_ -> zeros(Float64, cap), 6)
    GC.@preserve a demcmc_check(ccall((:demcmc_power_posterior, LIBDEMCMC), Cint,
        (Ptr{Cvoid}, Int64, Int64, Int32, Ref{CEvidence}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
        h, row0, n_rows, cap, ev, a[1], a[2], a[3], a[4], a[5], a[6]))
    K = Int(ev[].n_rungs)
    return (log_z_ti = ev[].log_z_ti, log_z_ti2 = ev[].log_z_ti2, log_z_ss = ev[].log_z_ss, se_ti = ev[].se_ti, se_ss = ev[].se_ss,
            t = a[1][1:K], mean_ll = a[2][1:K], var_ll = a[3][1:K], ess_ll = a[4][1:K], rhat_ll = a[5][1:K], log_ratio = a[6][1:K])
end

# Thermodynamic integration and stepping stones in ONE run: rung k is de.n_groups groups at t_k = (k / (K - 1))^power, all
# K rungs in one handle of K * de.n_groups groups (de.α must be 0: migration would move particles between temperatures).
# Returns the estimates and the t = 1 rung's chains.
function power_posterior(model::DEModel{<:GPULoglike}, de::DE, n_iter::Int; temperatures = nothing, n_temperatures = 32,
                         power = 5.0, device = 0, seed = rand(UInt64))
    t = temperatures === nothing ? [(k / (n_temperatures - 1))^power for k = 0:(n_temperatures - 1)] : Vector{Float64}(temperatures)
    de.α > 0 && throw(ArgumentError("power_posterior runs every rung as groups of one handle: pass DE(α = 0)"))
    G = de.n_groups
    job = deepcopy(de)
    job.n_groups = length(t) * G
    ev = Ref{Any}(nothing)
    chains = _sample_gpu(model, job, n_iter; device, seed, temperatures = repeat(t, inner = G), evidence = ev)
    top = (size(chains, 3) - G * de.Np + 1):size(chains, 3)
    return merge(ev[], (chains = chains[:, :, top],))
end
