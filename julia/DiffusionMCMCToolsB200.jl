#=
DiffusionMCMCToolsB200.jl — Julia glue over libdmt.so (include/dmt.h).

NOT EXECUTED IN THIS REPOSITORY'S CI: neither the build container nor the GPU box has Julia (SURVEY.md §0.7), so this file
is reviewed by eye only (the field names it reads off GuidedProposals' GuidProp and ObservationSchemes' LinearGsnObs objects —
P_target, P_aux, obs, L, Σ, t — are those of the versions pinned in /root/reference/Manifest.toml); the identical sequence of C calls is exercised from Python (diffusionmcmctools.jl_b200/_lib.py,
host.py) in tests/.  It adds device-backed methods to the reference's own generic functions, so a user loop written against
DiffusionMCMCTools.jl (docs/src/tutorials/block_ensemble/inference.md:44-75) runs unchanged on a `DeviceBlockEnsemble`.

Layout conversion: the reference stores one Trajectory per interval with cumulative Wiener paths; the library takes
X[point, dim, chain] and Wiener INCREMENTS W[step, dw, chain] with the chain index fastest (Julia arrays of size
(M, d, NP) / (M, dw, S), column-major).
=#
module DiffusionMCMCToolsB200

using DiffusionMCMCTools
import DiffusionMCMCTools: draw_proposal_path!, accept_reject_proposal_path!, swap_paths!, swap_XX!, swap_WW!, swap_PP!,
    swap_ll!, loglikhd!, loglikhd°!, fetch_ll, fetch_ll°, save_ll!, accpt_rate, ll_of_accepted, find_W_for_X!, set_proposal_law!,
    set_accepted!, set_ll!, recompute_path!
import GuidedProposals
import DiffusionDefinition
import ObservationSchemes
using StaticArrays
const GP = GuidedProposals
const DD = DiffusionDefinition
const OBS = ObservationSchemes

const libdmt = get(ENV, "DMT_LIB", joinpath(@__DIR__, "..", "diffusionmcmctools.jl_b200", "libdmt.so"))

# mirrors `dmt_config` (include/dmt.h)
struct DmtConfig
    model::Int32; n_chains::Int32; n_psets::Int32; n_intervals::Int32; obs_dim::Int32; device::Int32
    two_sided_laws::Int32; ll_hist_len::Int32; n_layouts::Int32; chain_offset::Int32; seed::UInt64; artificial_noise::Float64
end

struct DmtError <: Exception
    code::Int32
    msg::String
end

function check(ctx::Ptr{Cvoid}, rc::Int32)
    rc == 0 && return
    msg = unsafe_string(ccall((:dmt_last_error, libdmt), Cstring, (Ptr{Cvoid},), ctx))
    throw(DmtError(rc, msg))
end

"""
    DeviceEnsemble(model_id, theta, L, Σ, v, xbar, x0, n_pts, tt; kwargs...)

Device-resident `SamplingEnsemble` (src/sampling_ensemble.jl:17-41).  `v::Array{Float64,3}` is (P, m, K), `xbar` (P, d, K),
`x0` (M, d): chain / pset index fastest.
"""
mutable struct DeviceEnsemble
    ctx::Ptr{Cvoid}
    M::Int; P::Int; K::Int; d::Int; dw::Int
    next_layout::Int32
    theta::Matrix{Float64}      # (P, npar) accepted
    theta°::Matrix{Float64}
    xbar::Array{Float64,3}
    n_pts::Vector{Int32}        # points per observation interval
    tt::Vector{Float64}         # the imputation grid, interval after interval
end

function DeviceEnsemble(model::Integer, theta::Matrix{Float64}, L::Matrix{Float64}, Σ::Matrix{Float64}, v::Array{Float64,3},
                        xbar::Array{Float64,3}, x0::Matrix{Float64}, n_pts::Vector{Int32}, tt::Vector{Float64};
                        device=0, seed=UInt64(0), two_sided_laws=true, max_layouts=8, chain_offset=0, artificial_noise=1e-11)
    M, d = size(x0); P = size(v, 1); m = size(L, 1); K = length(n_pts)
    cfg = Ref(DmtConfig(model, M, P, K, m, device, two_sided_laws, 0, max_layouts, chain_offset, seed, artificial_noise))
    out = Ref{Ptr{Cvoid}}(C_NULL)
    rc = ccall((:dmt_create, libdmt), Int32, (Ref{DmtConfig}, Ptr{Int32}, Ptr{Float64}, Ptr{Int32}, Ref{Ptr{Cvoid}}),
               cfg, n_pts, tt, C_NULL, out)
    rc == 0 || throw(DmtError(rc, unsafe_string(ccall((:dmt_last_error, libdmt), Cstring, (Ptr{Cvoid},), C_NULL))))
    ctx = out[]
    dw = Ref{Int32}(0)
    ccall((:dmt_model_dims, libdmt), Int32, (Int32, Ptr{Int32}, Ref{Int32}, Ptr{Int32}, Ptr{Int32}), model, C_NULL, dw, C_NULL, C_NULL)
    # per-interval broadcast of L and Σ: [k][m*d][P] with P fastest
    Lk = repeat(reshape(permutedims(L), 1, d * m, 1), P, 1, K)          # row-major L flattened, (P, m*d, K)
    Σk = repeat(reshape(permutedims(Σ), 1, m * m, 1), P, 1, K)
    for side in (two_sided_laws ? (0, 1) : (0,))
        check(ctx, ccall((:dmt_set_params, libdmt), Int32, (Ptr{Cvoid}, Int32, Int32, Int32, Int32, Ptr{Float64}), ctx, side, 3, 0, K - 1, theta))
        check(ctx, ccall((:dmt_set_obs, libdmt), Int32, (Ptr{Cvoid}, Int32, Int32, Int32, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                         ctx, side, 0, K - 1, Lk, Σk, v))
        for store in (0, 1)   # aux_laws_blocking = aux_laws (src/sampling_unit.jl:57)
            check(ctx, ccall((:dmt_set_aux_linearised, libdmt), Int32, (Ptr{Cvoid}, Int32, Int32, Int32, Int32, Ptr{Float64}),
                             ctx, side, store, 0, K - 1, xbar))
        end
    end
    check(ctx, ccall((:dmt_set_start, libdmt), Int32, (Ptr{Cvoid}, Ptr{Float64}), ctx, x0))
    se = DeviceEnsemble(ctx, M, P, K, d, dw[], 0, copy(theta), copy(theta), xbar, copy(n_pts), copy(tt))
    finalizer(s -> ccall((:dmt_destroy, libdmt), Int32, (Ptr{Cvoid},), s.ctx), se)
    se
end

"""
    DeviceBlockEnsemble(se, block_ranges, ρρ=0.0, ll_hist_len=0)

`BlockEnsemble` (src/block_ensemble.jl:17-34) as one registered layout; `block_ranges` are the reference's 1-based UnitRanges.
"""
struct DeviceBlockEnsemble
    se::DeviceEnsemble
    layout::Int32
    n_blocks::Int
    ll_hist_len::Int
    ranges::Vector{UnitRange{Int}}   # the reference's 1-based interval ranges, one per block
end

function DeviceBlockEnsemble(se::DeviceEnsemble, block_ranges, ρρ=0.0, ll_hist_len=0)
    nb = length(block_ranges)
    i0 = Int32[first(r) - 1 for r in block_ranges]; i1 = Int32[last(r) - 1 for r in block_ranges]
    ρ = ρρ isa Number ? fill(Float64(ρρ), nb) : Vector{Float64}(ρρ)
    layout = se.next_layout; se.next_layout += 1
    check(se.ctx, ccall((:dmt_set_blocks, libdmt), Int32, (Ptr{Cvoid}, Int32, Int32, Ptr{Int32}, Ptr{Int32}, Ptr{Float64}, Ptr{UInt8}, Int32),
                        se.ctx, layout, nb, i0, i1, ρ, C_NULL, ll_hist_len))
    DeviceBlockEnsemble(se, layout, nb, ll_hist_len, [first(r):last(r) for r in block_ranges])
end

const DBE = DeviceBlockEnsemble

# ---- imputation (src/block_ensemble.jl:50,63-67).  mcmciter is 1-based in the reference, 0-based in the library.
draw_proposal_path!(be::DBE, mcmciter::Integer=1) =
    check(be.se.ctx, ccall((:dmt_draw_proposal_path, libdmt), Int32, (Ptr{Cvoid}, Int32, UInt32, Ptr{Float64}), be.se.ctx, be.layout, mcmciter - 1, C_NULL))
accept_reject_proposal_path!(be::DBE, mcmciter::Integer) =
    check(be.se.ctx, ccall((:dmt_accept_reject_path, libdmt), Int32, (Ptr{Cvoid}, Int32, UInt32, Ptr{Float64}), be.se.ctx, be.layout, mcmciter - 1, C_NULL))

# ---- swaps (src/block_ensemble.jl:79-112)
_swap(be::DBE, what) = check(be.se.ctx, ccall((:dmt_swap, libdmt), Int32, (Ptr{Cvoid}, Int32, Int32, Ptr{UInt8}), be.se.ctx, be.layout, what, C_NULL))
swap_XX!(be::DBE) = _swap(be, 1)
swap_WW!(be::DBE) = _swap(be, 2)
swap_paths!(be::DBE) = _swap(be, 3)
swap_ll!(be::DBE) = _swap(be, 8)
function swap_PP!(be::DBE)
    _swap(be, 4)
    be.se.theta, be.se.theta° = be.se.theta°, be.se.theta
    nothing
end

# ---- utility (src/block_ensemble.jl:121-179)
loglikhd!(be::DBE; skip=0) = check(be.se.ctx, ccall((:dmt_loglikhd, libdmt), Int32, (Ptr{Cvoid}, Int32, Int32, Int32), be.se.ctx, be.layout, 0, skip))
loglikhd°!(be::DBE; skip=0) = check(be.se.ctx, ccall((:dmt_loglikhd, libdmt), Int32, (Ptr{Cvoid}, Int32, Int32, Int32), be.se.ctx, be.layout, 1, skip))
function _stats(be::DBE)
    out = Vector{Float64}(undef, 2 + be.n_blocks)
    check(be.se.ctx, ccall((:dmt_allreduce_stats, libdmt), Int32, (Ptr{Cvoid}, Int32, Ptr{Float64}), be.se.ctx, be.layout, out))
    out
end
fetch_ll(be::DBE) = _stats(be)[1]
fetch_ll°(be::DBE) = _stats(be)[2]
save_ll!(be::DBE, i::Integer) = check(be.se.ctx, ccall((:dmt_save_ll, libdmt), Int32, (Ptr{Cvoid}, Int32, UInt32), be.se.ctx, be.layout, i - 1))
function accpt_rate(be::DBE, range)
    counts = Vector{Int64}(undef, be.n_blocks)
    check(be.se.ctx, ccall((:dmt_accept_counts, libdmt), Int32, (Ptr{Cvoid}, Int32, UInt32, UInt32, Ptr{Int64}),
                           be.se.ctx, be.layout, first(range) - 1, last(range) - 1, counts))
    counts ./ (length(range) * be.se.M)
end
function ll_of_accepted(be::DBE, i::Integer)
    n = be.n_blocks * be.se.M
    acc = Vector{UInt8}(undef, n); ll = Vector{Float64}(undef, n); ll° = Vector{Float64}(undef, n)
    check(be.se.ctx, ccall((:dmt_get_accept_history, libdmt), Int32, (Ptr{Cvoid}, Int32, UInt32, UInt32, Ptr{UInt8}), be.se.ctx, be.layout, i - 1, i - 1, acc))
    check(be.se.ctx, ccall((:dmt_get_ll_history, libdmt), Int32, (Ptr{Cvoid}, Int32, Int32, UInt32, UInt32, Ptr{Float64}), be.se.ctx, be.layout, 0, i - 1, i - 1, ll))
    check(be.se.ctx, ccall((:dmt_get_ll_history, libdmt), Int32, (Ptr{Cvoid}, Int32, Int32, UInt32, UInt32, Ptr{Float64}), be.se.ctx, be.layout, 1, i - 1, i - 1, ll°))
    reshape(ifelse.(acc .!= 0, ll°, ll), be.se.M, be.n_blocks)
end

# ---- blocking (src/block_ensemble.jl:192-221)
GP.set_obs!(be::DBE) = check(be.se.ctx, ccall((:dmt_set_artificial_obs, libdmt), Int32, (Ptr{Cvoid}, Int32), be.se.ctx, be.layout))
_rgt(be::DBE, which) = check(be.se.ctx, ccall((:dmt_recompute_guiding_term, libdmt), Int32, (Ptr{Cvoid}, Int32, Int32), be.se.ctx, be.layout, which))
GP.recompute_guiding_term!(be::DBE) = _rgt(be, 3)
GP.recompute_guiding_term!(be::DBE, ::Val{:P_only}) = _rgt(be, 1)
GP.recompute_guiding_term!(be::DBE, ::Val{:P°_only}) = _rgt(be, 2)
find_W_for_X!(be::DBE) = check(be.se.ctx, ccall((:dmt_find_W_for_X, libdmt), Int32, (Ptr{Cvoid}, Int32), be.se.ctx, be.layout))

# ---- the blocking step of docs/src/tutorials/block_collection/inference_with_blocking.md as one call:
# set_obs!; recompute_guiding_term!(Val(:P_only)); find_W_for_X!; loglikhd!; draw_proposal_path!
blocking_sweep!(be::DBE, mcmciter::Integer) =
    check(be.se.ctx, ccall((:dmt_blocking_sweep, libdmt), Int32, (Ptr{Cvoid}, Int32, UInt32), be.se.ctx, be.layout, mcmciter - 1))
# while θ, the auxiliary laws and the real observations stay fixed, K1 after set_obs! is F = F⁰ + Ψv (exact); see include/dmt.h
enable_guiding_cache!(be::DBE, on::Bool=true) =
    check(be.se.ctx, ccall((:dmt_enable_guiding_cache, libdmt), Int32, (Ptr{Cvoid}, Int32, Int32), be.se.ctx, be.layout, on))

# lanes per (chain, block) in the forward kernel: 0 = automatic (results never depend on it)
set_fwd_lanes!(se::DeviceEnsemble, lanes::Integer) =
    check(se.ctx, ccall((:dmt_set_fwd_lanes, libdmt), Int32, (Ptr{Cvoid}, Int32), se.ctx, lanes))
# multi-GPU, one process per GPU: export the 64-byte handle, all-gather it (MPI.Allgather, Distributed, ...), map the peers
p2p_export(se::DeviceEnsemble) = (h = zeros(UInt8, 64);
    check(se.ctx, ccall((:dmt_p2p_export, libdmt), Int32, (Ptr{Cvoid}, Ptr{UInt8}), se.ctx, h)); h)
p2p_init!(se::DeviceEnsemble, n_ranks::Integer, rank::Integer, handles::Matrix{UInt8}) =   # handles: 64 x n_ranks
    check(se.ctx, ccall((:dmt_p2p_init, libdmt), Int32, (Ptr{Cvoid}, Int32, Int32, Ptr{UInt8}), se.ctx, n_ranks, rank, handles))

# ---- parameters (src/block_ensemble.jl:242-255 -> src/biblock.jl:334-371).  The name translation of
# src/param_names_collections.jl stays here on the host: `pnames` is its result for the target law,
# a vector of (index into θ°) => (index into the model's parameter vector) pairs.
function set_proposal_law!(be::DBE, θ°, pnames::Vector{Pair{Int,Int}}, critical_change::Bool; skip=0)
    se = be.se
    th = copy(se.theta)
    for (i, j) in pnames
        th[:, j] .= θ°[i]
    end
    se.theta° = th
    # GP.equalize_obs_params! / equalize_law_params! FIRST (src/biblock.jl:362-363): b° := b for every record; when b° had to be changed its
    # guiding term belongs to other parameters, and the update is escalated to a critical one exactly like the reference does
    changed = Ref{Int32}(0)
    check(se.ctx, ccall((:dmt_equalize_laws, libdmt), Int32, (Ptr{Cvoid}, Int32, Int32, Int32, Ref{Int32}), se.ctx, 3, 0, se.K - 1, changed))
    critical_change = critical_change || changed[] != 0
    check(se.ctx, ccall((:dmt_set_params, libdmt), Int32, (Ptr{Cvoid}, Int32, Int32, Int32, Int32, Ptr{Float64}), se.ctx, 1, 3, 0, se.K - 1, th))
    # Auxiliary laws evaluated on the HOST (DeviceEnsemble built from a SamplingEnsemble): a critical update changes them, and only the
    # reference's own objects know how — update those (DD.set_parameters! on the host proposal laws) and call upload_aux!(se, se_host, 1)
    # BEFORE this function; nothing to do here.  Device-linearised auxiliary laws (raw-array constructor) are re-linearised below.
    if critical_change && !isempty(se.xbar)
        for store in (0, 1)   # the linearisation points are already on the device: NULL re-linearises there with the new θ°
            check(se.ctx, ccall((:dmt_set_aux_linearised, libdmt), Int32, (Ptr{Cvoid}, Int32, Int32, Int32, Int32, Ptr{Float64}),
                                se.ctx, 1, store, 0, se.K - 1, C_NULL))
        end
    end
    check(se.ctx, ccall((:dmt_set_proposal_law, libdmt), Int32, (Ptr{Cvoid}, Int32, Int32, Int32), se.ctx, be.layout, critical_change, skip))
end

# ---- paths back into the reference's containers -------------------------------------------------------------------------
# The library's natural layout is X[point, dim, chain] (C order), i.e. a Julia array of size (M, d, NP), and Wiener INCREMENTS
# W[step, dw, chain] = (M, dw, S).  The reference keeps, per recording and observation interval, a Trajectory of states on the interval's
# grid (first point = last point of the previous interval) and a Trajectory of the cumulative Wiener path starting at 0.
_npts(se::DeviceEnsemble) = se.n_pts
_pt0(se::DeviceEnsemble) = cumsum(vcat(0, se.n_pts))                     # 0-based first point of interval k (k = 1..K at index k)
_step0(se::DeviceEnsemble) = cumsum(vcat(0, se.n_pts .- 1))

"""    get_X(se, side=0) -> Array{Float64,3} of size (M, d, NP);  get_W(se, side=0) -> (M, dw, S)   (`bb.b.XX`, `bb.b.WW` of every recording)"""
function get_X(se::DeviceEnsemble, side::Integer=0)
    X = Array{Float64,3}(undef, se.M, se.d, sum(se.n_pts))
    check(se.ctx, ccall((:dmt_get_X, libdmt), Int32, (Ptr{Cvoid}, Int32, Ptr{Float64}), se.ctx, side, X))
    X
end
function get_W(se::DeviceEnsemble, side::Integer=0)
    W = Array{Float64,3}(undef, se.M, se.dw, sum(se.n_pts) - se.K)
    check(se.ctx, ccall((:dmt_get_W, libdmt), Int32, (Ptr{Cvoid}, Int32, Ptr{Float64}), se.ctx, side, W))
    W
end
"""paths / noise of the listed recordings only (1-based): (length(recs), d, NP) and (length(recs), dw, S)"""
function get_X(se::DeviceEnsemble, recs::AbstractVector{<:Integer}, side::Integer=0)
    sel = Int32.(recs .- 1)
    X = Array{Float64,3}(undef, length(sel), se.d, sum(se.n_pts))
    check(se.ctx, ccall((:dmt_get_X_chains, libdmt), Int32, (Ptr{Cvoid}, Int32, Int32, Ptr{Int32}, Ptr{Float64}), se.ctx, side, length(sel), sel, X))
    X
end
function get_W(se::DeviceEnsemble, recs::AbstractVector{<:Integer}, side::Integer=0)
    sel = Int32.(recs .- 1)
    W = Array{Float64,3}(undef, length(sel), se.dw, sum(se.n_pts) - se.K)
    check(se.ctx, ccall((:dmt_get_W_chains, libdmt), Int32, (Ptr{Cvoid}, Int32, Int32, Ptr{Int32}, Ptr{Float64}), se.ctx, side, length(sel), sel, W))
    W
end

"""
    trajectories(se, X, r, intervals=1:se.K) -> Vector{Trajectory}

Row `r` of a `get_X` result as the reference's `XX`: one `Trajectory(t, x::Vector{SVector{d}})` per observation interval
(`src/sampling_unit.jl:66` `XX, WW = trajectory(PP)`).
"""
function trajectories(se::DeviceEnsemble, X::Array{Float64,3}, r::Integer, intervals=1:se.K)
    p0 = _pt0(se)
    map(intervals) do k
        idx = (p0[k] + 1):p0[k + 1]
        DD.Trajectory(se.tt[idx], [SVector{se.d,Float64}(ntuple(i -> X[r, i, j], se.d)) for j in idx])
    end
end
"""the same for the noise: increments -> cumulative Wiener path starting at zero on each interval (`WW[k].x[1] == 0`)"""
function wiener_trajectories(se::DeviceEnsemble, W::Array{Float64,3}, r::Integer, intervals=1:se.K)
    p0, s0 = _pt0(se), _step0(se)
    map(intervals) do k
        w = zeros(SVector{se.dw,Float64}, se.n_pts[k])
        for (n, j) in enumerate((s0[k] + 1):s0[k + 1])
            w[n + 1] = w[n] + SVector{se.dw,Float64}(ntuple(i -> W[r, i, j], se.dw))
        end
        DD.Trajectory(se.tt[(p0[k] + 1):p0[k + 1]], w)
    end
end
"""    get_paths(se, side=0) -> Vector{Vector{Trajectory}}: `[deepcopy(rec.u.XX) for rec in se.recordings]` of the tutorials' save step"""
function get_paths(se::DeviceEnsemble, side::Integer=0)
    X = get_X(se, side)
    [trajectories(se, X, r) for r in 1:se.M]
end
"""the inverse converters (upload host containers): `XX::Vector{Vector{Trajectory}}` -> (M, d, NP); cumulative `WW` -> increments (M, dw, S)"""
function pack_paths(se::DeviceEnsemble, XXs)
    X = Array{Float64,3}(undef, se.M, se.d, sum(se.n_pts)); p0 = _pt0(se)
    for r in 1:se.M, k in 1:se.K, (n, j) in enumerate((p0[k] + 1):p0[k + 1]), i in 1:se.d
        X[r, i, j] = XXs[r][k].x[n][i]
    end
    X
end
function pack_noise(se::DeviceEnsemble, WWs)
    W = Array{Float64,3}(undef, se.M, se.dw, sum(se.n_pts) - se.K); s0 = _step0(se)
    for r in 1:se.M, k in 1:se.K, (n, j) in enumerate((s0[k] + 1):s0[k + 1]), i in 1:se.dw
        W[r, i, j] = WWs[r][k].x[n + 1][i] - WWs[r][k].x[n][i]
    end
    W
end
set_X!(se::DeviceEnsemble, X::Array{Float64,3}, side::Integer=0) = check(se.ctx, ccall((:dmt_set_X, libdmt), Int32, (Ptr{Cvoid}, Int32, Ptr{Float64}), se.ctx, side, X))
set_W!(se::DeviceEnsemble, W::Array{Float64,3}, side::Integer=0) = check(se.ctx, ccall((:dmt_set_W, libdmt), Int32, (Ptr{Cvoid}, Int32, Ptr{Float64}), se.ctx, side, W))

# ---- the reference's constructor -------------------------------------------------------------------------------------------
# SamplingEnsemble(aux_laws, recordings, tts, args...; aux_laws_blocking, artificial_noise, solver_choice_blocking)
# (src/sampling_ensemble.jl:20-40).  The device ensemble is built FROM the host ensemble the reference's own constructor returns: the
# target law's parameters, the observation operators and the auxiliary laws' (B, β, σ̃) are read off its GuidProp objects — so ANY
# auxiliary law the user passes works (its coefficients are evaluated by the reference's own code and uploaded with dmt_set_aux) — and
# the initial paths are the ones `init_paths!` drew on the host (src/sampling_unit.jl:70), uploaded with dmt_set_X / dmt_set_W.
const MODEL_IDS = Dict(:FitzHughNagumo => 0, :LotkaVolterra => 1, :Lorenz => 2, :Prokaryote => 3, :JansenRit => 4)
const PARAM_ORDER = Dict(                                    # order of theta in include/dmt.h
    :FitzHughNagumo => [:ϵ, :s, :γ, :β, :σ], :LotkaVolterra => [:α, :β, :γ, :δ, :σ1, :σ2], :Lorenz => [:θ₁, :θ₂, :θ₃, :σ],
    :Prokaryote => [:c₁, :c₂, :c₃, :c₄, :c₅, :c₆, :c₇, :c₈, :K], :JansenRit => [:A, :a, :B, :b, :C, :νmax, :v0, :r, :μy, :σy])

function DeviceEnsemble(se_host::SamplingEnsemble; device=0, seed=UInt64(0), two_sided_laws=true, max_layouts=8, chain_offset=0,
                        artificial_noise=1e-11, model=nothing, θnames=nothing)
    recs = se_host.recordings
    M = length(recs); u1 = recs[1].u
    K = length(u1.PP)
    Pt = u1.PP[1].P_target
    mname = nameof(typeof(Pt))
    model_id = model === nothing ? MODEL_IDS[mname] : model
    names = θnames === nothing ? PARAM_ORDER[mname] : θnames
    d = DD.dimension(Pt).process
    n_pts = Int32[length(u1.XX[k].t) for k in 1:K]
    tt = vcat((u1.XX[k].t for k in 1:K)...)
    m = length(u1.PP[1].obs.obs)
    # every recording must live on the same grid with the same observation dimension (else: one DeviceEnsemble per bucket, hetero.py)
    all(r -> length(r.u.PP) == K && all(k -> r.u.XX[k].t == u1.XX[k].t, 1:K), recs) ||
        error("recordings differ in their time grids: bucket them (see hetero.py) and build one DeviceEnsemble per bucket")
    theta = [Float64(getfield(recs[r].u.PP[1].P_target, nm)) for r in 1:M, nm in names]                  # (P = M, npar)
    Lk = Array{Float64,3}(undef, M, m * d, K); Σk = Array{Float64,3}(undef, M, m * m, K); v = Array{Float64,3}(undef, M, m, K)
    x0 = [recs[r].u.XX[1].x[1][i] for r in 1:M, i in 1:d]
    cfg = Ref(DmtConfig(model_id, M, M, K, m, device, two_sided_laws, 0, max_layouts, chain_offset, seed, artificial_noise))
    out = Ref{Ptr{Cvoid}}(C_NULL)
    rc = ccall((:dmt_create, libdmt), Int32, (Ref{DmtConfig}, Ptr{Int32}, Ptr{Float64}, Ptr{Int32}, Ref{Ptr{Cvoid}}), cfg, n_pts, tt, C_NULL, out)
    rc == 0 || throw(DmtError(rc, unsafe_string(ccall((:dmt_last_error, libdmt), Cstring, (Ptr{Cvoid},), C_NULL))))
    ctx = out[]
    dw = Ref{Int32}(0)
    ccall((:dmt_model_dims, libdmt), Int32, (Int32, Ptr{Int32}, Ref{Int32}, Ptr{Int32}, Ptr{Int32}), model_id, C_NULL, dw, C_NULL, C_NULL)
    # auxiliary laws, evaluated by the reference: B [k][d*d][P] row-major, β [k][d][P], ã = σ̃σ̃' [k][d*d][P]
    function aux_arrays(getlaws)
        B = Array{Float64,3}(undef, M, d * d, K); β = Array{Float64,3}(undef, M, d, K); a = Array{Float64,3}(undef, M, d * d, K)
        for r in 1:M, k in 1:K
            P̃ = getlaws(recs[r])[k].P_aux; t = u1.XX[k].t[1]
            Bm = DD.B(t, P̃); βv = DD.β(t, P̃); σm = DD.σ(t, P̃); am = σm * σm'
            for i in 1:d, j in 1:d
                B[r, (i - 1) * d + j, k] = Bm[i, j]; a[r, (i - 1) * d + j, k] = am[i, j]
            end
            for i in 1:d
                β[r, i, k] = βv[i]
            end
        end
        B, β, a
    end
    for r in 1:M, k in 1:K
        o = recs[r].u.PP[k].obs
        for a in 1:m, j in 1:d
            Lk[r, (a - 1) * d + j, k] = o.L[a, j]
        end
        for a in 1:m, b in 1:m
            Σk[r, (a - 1) * m + b, k] = o.Σ[a, b]
        end
        for a in 1:m
            v[r, a, k] = o.obs[a]
        end
    end
    B, β, a = aux_arrays(r -> r.u.PP); Bb, βb, ab = aux_arrays(r -> r.u.PPb)
    for side in (two_sided_laws ? (0, 1) : (0,))
        check(ctx, ccall((:dmt_set_params, libdmt), Int32, (Ptr{Cvoid}, Int32, Int32, Int32, Int32, Ptr{Float64}), ctx, side, 3, 0, K - 1, theta))
        check(ctx, ccall((:dmt_set_obs, libdmt), Int32, (Ptr{Cvoid}, Int32, Int32, Int32, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}), ctx, side, 0, K - 1, Lk, Σk, v))
        check(ctx, ccall((:dmt_set_aux, libdmt), Int32, (Ptr{Cvoid}, Int32, Int32, Int32, Int32, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}), ctx, side, 0, 0, K - 1, B, β, a))
        check(ctx, ccall((:dmt_set_aux, libdmt), Int32, (Ptr{Cvoid}, Int32, Int32, Int32, Int32, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}), ctx, side, 1, 0, K - 1, Bb, βb, ab))
    end
    check(ctx, ccall((:dmt_set_start, libdmt), Int32, (Ptr{Cvoid}, Ptr{Float64}), ctx, x0))
    se = DeviceEnsemble(ctx, M, M, K, d, dw[], 0, copy(theta), copy(theta), zeros(0, 0, 0), n_pts, tt)
    finalizer(s -> ccall((:dmt_destroy, libdmt), Int32, (Ptr{Cvoid},), s.ctx), se)
    # the paths init_paths! drew on the host (u and u° = deepcopy(u), src/sampling_pair.jl:51)
    X = pack_paths(se, [r.u.XX for r in recs]); W = pack_noise(se, [r.u.WW for r in recs])
    for side in (0, 1)
        set_X!(se, X, side); set_W!(se, W, side)
    end
    se
end
"""
    upload_aux!(se, se_host, side; proposal=(side == 1))

Re-evaluate `(B, β, σ̃σ̃')` of the host ensemble's CURRENT auxiliary laws (`u` or `u°`, both stores) with the reference's own code and upload
them to law side `side` — what a critical parameter update needs when the auxiliary laws are host-evaluated.
"""
function upload_aux!(se::DeviceEnsemble, se_host::SamplingEnsemble, side::Integer; proposal::Bool=(side == 1))
    recs = se_host.recordings; M, K, d = se.M, se.K, se.d
    for (store, field) in ((0, :PP), (1, :PPb))
        B = Array{Float64,3}(undef, M, d * d, K); β = Array{Float64,3}(undef, M, d, K); a = Array{Float64,3}(undef, M, d * d, K)
        for r in 1:M, k in 1:K
            u = proposal ? recs[r].u° : recs[r].u
            P̃ = getfield(u, field)[k].P_aux; t = se.tt[_pt0(se)[k] + 1]
            Bm = DD.B(t, P̃); βv = DD.β(t, P̃); σm = DD.σ(t, P̃); am = σm * σm'
            for i in 1:d, j in 1:d
                B[r, (i - 1) * d + j, k] = Bm[i, j]; a[r, (i - 1) * d + j, k] = am[i, j]
            end
            for i in 1:d
                β[r, i, k] = βv[i]
            end
        end
        check(se.ctx, ccall((:dmt_set_aux, libdmt), Int32, (Ptr{Cvoid}, Int32, Int32, Int32, Int32, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                            se.ctx, side, store, 0, K - 1, B, β, a))
    end
end
DeviceEnsemble(aux_laws, recordings, tts, args=tuple(); device=0, seed=UInt64(0), two_sided_laws=true, max_layouts=8, chain_offset=0, kwargs...) =
    DeviceEnsemble(SamplingEnsemble(aux_laws, recordings, tts, args; kwargs...); device=device, seed=seed, two_sided_laws=two_sided_laws,
                   max_layouts=max_layouts, chain_offset=chain_offset, artificial_noise=get(kwargs, :artificial_noise, 1e-11))
OBS.num_recordings(se::DeviceEnsemble) = se.M
OBS.num_recordings(be::DBE) = be.se.M

# ---- saving while sampling: thinned paths and history chunks leave on a second stream (include/dmt.h) ----------------------
# `paths[i ÷ 400] = deepcopy(bb.b.XX)` of the tutorials / reading b.ll_history at the end.  Buffers must stay alive (and should be
# page-locked) until `snapshot_wait(se)` returns.
snapshot_paths_async!(out::Array{Float64,3}, se::DeviceEnsemble, recs::AbstractVector{<:Integer}, side::Integer=0) =   # out: (length(recs), d, NP)
    check(se.ctx, ccall((:dmt_snapshot_paths_async, libdmt), Int32, (Ptr{Cvoid}, Int32, Int32, Ptr{Int32}, Ptr{Float64}), se.ctx, side, length(recs), Int32.(recs .- 1), out))
histories_async!(ll::Array{Float64,4}, acc::Array{UInt8,3}, be::DBE, range) =                                            # ll: (M, n_blocks, 2, n), acc: (M, n_blocks, n)
    check(be.se.ctx, ccall((:dmt_histories_async, libdmt), Int32, (Ptr{Cvoid}, Int32, UInt32, UInt32, Ptr{Float64}, Ptr{UInt8}),
                           be.se.ctx, be.layout, first(range) - 1, last(range) - 1, ll, acc))
snapshot_wait(se::DeviceEnsemble) = check(se.ctx, ccall((:dmt_snapshot_wait, libdmt), Int32, (Ptr{Cvoid},), se.ctx))

# ---- posterior summaries of the paths: per-recording running moments of the accepted path, on the device (include/dmt.h) -------
# The tutorials' `paths[i ÷ 400] = deepcopy(bb.b.XX)` (docs/src/tutorials/biblock/smoothing.md:55) summarised by mean and variance for
# every recording, without copying paths: call `path_moments_add!(se)` at each saving iteration, read the summaries at the end.
path_moments_add!(se::DeviceEnsemble) = check(se.ctx, ccall((:dmt_path_moments_add, libdmt), Int32, (Ptr{Cvoid},), se.ctx))
path_moments_reset!(se::DeviceEnsemble) = check(se.ctx, ccall((:dmt_path_moments_reset, libdmt), Int32, (Ptr{Cvoid},), se.ctx))
"""    path_moments(se, recs=1:se.M) -> (mean, var, count): mean and var of size (length(recs), d, NP), var = m2 / count"""
function path_moments(se::DeviceEnsemble, recs::AbstractVector{<:Integer}=1:se.M)
    sel = Int32.(recs .- 1)
    mean = Array{Float64,3}(undef, length(sel), se.d, sum(se.n_pts)); m2 = similar(mean); n = Ref{UInt64}(0)
    check(se.ctx, ccall((:dmt_get_path_moments, libdmt), Int32, (Ptr{Cvoid}, Int32, Ptr{Int32}, Ptr{Float64}, Ptr{Float64}, Ref{UInt64}),
                        se.ctx, length(sel), sel, mean, m2, n))
    mean, m2 ./ n[], Int(n[])
end
"""restore all recordings' moments from `mean`, `m2` (size (M, d, NP)) after `count` updates (checkpoint / resume)"""
set_path_moments!(se::DeviceEnsemble, mean::Array{Float64,3}, m2::Array{Float64,3}, count::Integer) =
    check(se.ctx, ccall((:dmt_set_path_moments, libdmt), Int32, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, UInt64), se.ctx, mean, m2, count))
"""    pset_path_moments(se) -> (mean, var, rhat), each (P, d, NP): pooled over the recordings that share a data set; Gelman-Rubin R-hat"""
function pset_path_moments(se::DeviceEnsemble)
    mean = Array{Float64,3}(undef, se.P, se.d, sum(se.n_pts)); var = similar(mean); rhat = similar(mean)
    check(se.ctx, ccall((:dmt_get_pset_path_moments, libdmt), Int32, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}), se.ctx, mean, var, rhat))
    mean, var, rhat
end

# ---- BlockCollection / BiBlock views (src/block_collection.jl:17-36, src/biblock.jl:17-62) ---------------------------------
# `be.recordings[r]` and `.blocks[b]` of the reference.  The numerical calls are batched over all recordings and blocks on the device —
# call them on the DeviceBlockEnsemble; the views carry what acts on ONE recording / ONE block: reading XX, WW, ll and the histories,
# the swaps, set_accepted!, set_ll!, ll_of_accepted, accpt_rate.
struct DeviceBiBlock
    be::DBE; rec::Int; blk::Int
end
struct DeviceBlockCollection
    be::DBE; rec::Int
end
recordings(be::DBE) = [DeviceBlockCollection(be, r) for r in 1:be.se.M]
blocks(bc::DeviceBlockCollection) = [DeviceBiBlock(bc.be, bc.rec, b) for b in 1:bc.be.n_blocks]
Base.getindex(be::DBE, r::Integer) = DeviceBlockCollection(be, r)
Base.getindex(bc::DeviceBlockCollection, b::Integer) = DeviceBiBlock(bc.be, bc.rec, b)
_intervals(bb::DeviceBiBlock) = bb.be.ranges[bb.blk]
XX(bb::DeviceBiBlock, side::Integer=0) = trajectories(bb.be.se, get_X(bb.be.se, [bb.rec], side), 1, _intervals(bb))
WW(bb::DeviceBiBlock, side::Integer=0) = wiener_trajectories(bb.be.se, get_W(bb.be.se, [bb.rec], side), 1, _intervals(bb))
function _ll(be::DBE, side::Integer)
    ll = Matrix{Float64}(undef, be.se.M, be.n_blocks)
    check(be.se.ctx, ccall((:dmt_get_ll, libdmt), Int32, (Ptr{Cvoid}, Int32, Int32, Ptr{Float64}), be.se.ctx, be.layout, side, ll))
    ll
end
ll(bb::DeviceBiBlock, side::Integer=0) = _ll(bb.be, side)[bb.rec, bb.blk]
fetch_ll(bc::DeviceBlockCollection) = sum(_ll(bc.be, 0)[bc.rec, :])          # src/block_collection.jl:144
fetch_ll°(bc::DeviceBlockCollection) = sum(_ll(bc.be, 1)[bc.rec, :])         # src/block_collection.jl:156
function _swap_blocks(be::DBE, what, mask::Matrix{UInt8})                    # mask (M, n_blocks) == C [n_blocks][M]
    check(be.se.ctx, ccall((:dmt_swap_blocks, libdmt), Int32, (Ptr{Cvoid}, Int32, Int32, Ptr{UInt8}), be.se.ctx, be.layout, what, mask))
end
_mask(bb::DeviceBiBlock) = (m = zeros(UInt8, bb.be.se.M, bb.be.n_blocks); m[bb.rec, bb.blk] = 1; m)
_mask(bc::DeviceBlockCollection) = (m = zeros(UInt8, bc.be.se.M, bc.be.n_blocks); m[bc.rec, :] .= 1; m)
for (f, what) in ((:swap_XX!, 1), (:swap_WW!, 2), (:swap_paths!, 3), (:swap_ll!, 8), (:swap_PP!, 4))   # src/biblock.jl:148-209, src/block_collection.jl:84-118
    @eval $f(v::Union{DeviceBiBlock,DeviceBlockCollection}) = _swap_blocks(v.be, $what, _mask(v))
end
function _hist_row(be::DBE, i::Integer)
    n = be.n_blocks * be.se.M
    acc = Vector{UInt8}(undef, n)
    check(be.se.ctx, ccall((:dmt_get_accept_history, libdmt), Int32, (Ptr{Cvoid}, Int32, UInt32, UInt32, Ptr{UInt8}), be.se.ctx, be.layout, i - 1, i - 1, acc))
    reshape(acc, be.se.M, be.n_blocks)
end
function set_accepted!(bb::DeviceBiBlock, i::Integer, v::Bool)               # src/biblock.jl:130-135
    a = _hist_row(bb.be, i); a[bb.rec, bb.blk] = v
    check(bb.be.se.ctx, ccall((:dmt_set_accepted, libdmt), Int32, (Ptr{Cvoid}, Int32, UInt32, Ptr{UInt8}), bb.be.se.ctx, bb.be.layout, i - 1, a))
end
function set_ll!(bb::DeviceBiBlock, i::Integer, v::Real; side::Integer=0)   # set_ll!(bb.b, i, v)  src/block.jl:82-86
    be = bb.be; n = be.n_blocks * be.se.M
    h = Vector{Float64}(undef, n)
    check(be.se.ctx, ccall((:dmt_get_ll_history, libdmt), Int32, (Ptr{Cvoid}, Int32, Int32, UInt32, UInt32, Ptr{Float64}), be.se.ctx, be.layout, side, i - 1, i - 1, h))
    h[(bb.blk - 1) * be.se.M + bb.rec] = v
    check(be.se.ctx, ccall((:dmt_set_ll_history, libdmt), Int32, (Ptr{Cvoid}, Int32, Int32, UInt32, Ptr{Float64}), be.se.ctx, be.layout, side, i - 1, h))
end
# recompute_path!(b°, b.WW; skip) for every recording and block (src/block.jl:161-187): proposal law and X°, accepted noise
recompute_path!(be::DBE; skip=0, law_side=1, noise_side=0) =
    check(be.se.ctx, ccall((:dmt_recompute_path, libdmt), Int32, (Ptr{Cvoid}, Int32, Int32, Int32, Int32), be.se.ctx, be.layout, law_side, noise_side, skip))
accpt_rate(bb::DeviceBiBlock, range) = sum(_hist_row(bb.be, i)[bb.rec, bb.blk] for i in range) / length(range)   # src/biblock.jl:232
accpt_rate(bc::DeviceBlockCollection, range) = [accpt_rate(bb, range) for bb in blocks(bc)]                       # src/block_collection.jl:180-184
ll_of_accepted(bb::DeviceBiBlock, i::Integer) = ll_of_accepted(bb.be, i)[bb.rec, bb.blk]                          # src/biblock.jl:222-225
ll_of_accepted(bc::DeviceBlockCollection, i::Integer) = ll_of_accepted(bc.be, i)[bc.rec, :]                       # src/block_collection.jl:172

# ---- the pCN memory: one ρ per (recording, block) as in the reference (bb.ρ, src/biblock.jl:46), and its adaptation toward a
# target acceptance rate on the device (include/dmt.h).  Burn-in: blocking_sweep!; accept_reject_proposal_path!; adapt_rho!; then
# disable_rho_adaptation! before keeping samples (draws taken while ρ adapts are not from a fixed Markov kernel).
"""    rho_chains(be) -> Matrix (M, n_blocks): ρ of every block of every recording"""
function rho_chains(be::DBE)
    ρ = Matrix{Float64}(undef, be.se.M, be.n_blocks)
    check(be.se.ctx, ccall((:dmt_get_rho_chains, libdmt), Int32, (Ptr{Cvoid}, Int32, Ptr{Float64}), be.se.ctx, be.layout, ρ))
    ρ
end
"""    set_rho_chains!(be, ρ): ρ broadcasts to (M, n_blocks); on an adapting layout the adaptation restarts from the new values"""
function set_rho_chains!(be::DBE, ρ)
    r = Matrix{Float64}(undef, be.se.M, be.n_blocks)
    r .= ρ
    check(be.se.ctx, ccall((:dmt_set_rho_chains, libdmt), Int32, (Ptr{Cvoid}, Int32, Ptr{Float64}), be.se.ctx, be.layout, r))
end
enable_rho_adaptation!(be::DBE; target=0.234, γ0=1.0, decay=0.66, window=10, ρmin=0.0, ρmax=0.999) =
    check(be.se.ctx, ccall((:dmt_set_rho_adaptation, libdmt), Int32, (Ptr{Cvoid}, Int32, Float64, Float64, Float64, Int32, Float64, Float64),
                           be.se.ctx, be.layout, target, γ0, decay, window, ρmin, ρmax))
disable_rho_adaptation!(be::DBE) =
    check(be.se.ctx, ccall((:dmt_set_rho_adaptation, libdmt), Int32, (Ptr{Cvoid}, Int32, Float64, Float64, Float64, Int32, Float64, Float64),
                           be.se.ctx, be.layout, 0.0, 0.0, 0.0, 0, 0.0, 0.0))
adapt_rho!(be::DBE) = check(be.se.ctx, ccall((:dmt_adapt_rho, libdmt), Int32, (Ptr{Cvoid}, Int32), be.se.ctx, be.layout))
# bb.ρ reads and writes that one (recording, block) entry
Base.getproperty(bb::DeviceBiBlock, s::Symbol) =
    s === :ρ ? rho_chains(getfield(bb, :be))[getfield(bb, :rec), getfield(bb, :blk)] : getfield(bb, s)
function Base.setproperty!(bb::DeviceBiBlock, s::Symbol, v)
    s === :ρ || return setfield!(bb, s, v)
    be = getfield(bb, :be)
    r = rho_chains(be)
    r[getfield(bb, :rec), getfield(bb, :blk)] = v
    set_rho_chains!(be, r)
end

export DeviceEnsemble, DeviceBlockEnsemble, DeviceBlockCollection, DeviceBiBlock, upload_aux!, get_paths, get_X, get_W, trajectories,
    wiener_trajectories, pack_paths, pack_noise, recordings, blocks, blocking_sweep!, enable_guiding_cache!, path_moments_add!,
    path_moments_reset!, path_moments, set_path_moments!, pset_path_moments, rho_chains, set_rho_chains!, enable_rho_adaptation!,
    disable_rho_adaptation!, adapt_rho!

end # module
