# WSB200.jl — makes libwsb200.so (include/wsb200.h) the storage / kernel backend of WeightedSampling.jl.
#
#     using WeightedSampling, WSB200
#     @model function ssm(obs) ... end                    # the reference's OWN macro, unmodified
#     state = WSB200.DeviceSMCState(100_000_000; ess_perc_min = 1.0)
#     run!(ssm(obs), state)                               # every statement is one ccall; nothing runs on the CPU
#     WSB200.log_evidence(state), WSB200.expectation(x -> x, state)
#
# How the unmodified `@model` output runs here.  `@model` emits `Sample(:x, kernel, state -> (args...))`,
# `Observe(...)`, `Assign(...)`, ... whose argument closures are FUSED BROADCASTS over
# `getcol(state.store, :x)` (src/rewrites.jl:146-219: `vectorize`).  For a `DeviceColumnStore`, `getcol` returns a
# lazy handle (`DeviceVec`) with its own `BroadcastStyle`; materialising a broadcast over such handles does not compute
# anything, it SERIALISES the fused broadcast tree into the postfix tokens of include/wsb200.h (`lower`).  So
# `t.argfn(state)` hands the `apply!` methods below device expressions, the kernel object is matched BY IDENTITY
# against `WeightedSampling.default_kernels` (src/default_kernels.jl:83-102) to pick the device op, and a kernel or
# function outside the device-op set is an error (`UnsupportedModelError`), never a CPU fallback.
# `WSB200.@device_model` wraps `@model` and performs that check at macro-expansion time for the kernel names it can
# see.
#
# NOT EXECUTED IN THIS REPOSITORY'S CI: the build image has no Julia toolchain (`which julia` is empty, no network).
# The Python host (weightedsampling.jl_b200/) issues the same C-ABI call sequence and is what the tests drive;
# tests/host/abi_smoke.c drives it from plain C.  This file is the binding a maintainer of the reference would add
# (INTEGRATION.md walks through it).
module WSB200

using WeightedSampling
using Random
import WeightedSampling: AbstractParticleStore, SMCState, ParticleTransformer, WeightedKernel, nparticles, hascol,
    getcol, colnames, broadcast_setcol!, resample!, apply!, score!, run!, advance!, score_logpdf,
    Assign, Sample, AccessorSample, Observe, Weight, Resample, Move, Sequence, Loop, Cond, ScoreCtx

const LIB = get(ENV, "WSB200_LIB", joinpath(@__DIR__, "..", "weightedsampling.jl_b200", "lib", "libwsb200.so"))

struct UnsupportedModelError <: Exception
    msg::String
end
Base.showerror(io::IO, e::UnsupportedModelError) = print(io, "UnsupportedModelError: ", e.msg)
unsupported(msg) = throw(UnsupportedModelError(msg * " — outside the device-op set of libwsb200 (no CPU fallback)"))

# ---- include/wsb200.h mirrors ------------------------------------------------------------------------------------
struct WsTok
    op::Int32; col::Int32; comp::Int32; reserved::Int32; val::Float64
end
struct WsExpr
    toks::Ptr{WsTok}; n::Int32; reserved::Int32
end
struct WsResampleInfo
    fired::Int32; resampled::Int32; ess_perc::Float64; log_mean_w::Float64; n_clamped::Int64
end
WsResampleInfo() = WsResampleInfo(0, 0, NaN, NaN, 0)
struct WsMoveSpec
    n_targets::Int32; col::Ptr{Int32}; comp::Ptr{Int32}; proposal::Int32; has_bounds::Int32
    lo::Ptr{Float64}; hi::Ptr{Float64}; step::Float64; diversity::Float64; target_depth::Int64
end
struct WsMoveInfo
    ran::Int32; reserved::Int32; diversity::Float64; n_accepted::Int64
end
struct WsPlaneStats
    mean::Float64; median::Float64; std::Float64; min::Float64; max::Float64; hist::NTuple{8,Float64}
end

const TOK_CONST, TOK_PLANE, TOK_ADD, TOK_SUB, TOK_MUL, TOK_DIV, TOK_NEG, TOK_EXP, TOK_LOG, TOK_SQRT, TOK_SQUARE,
      TOK_SIN, TOK_COS, TOK_ABS, TOK_POW, TOK_RANDN, TOK_RANDU, TOK_RANDEXP, TOK_LT, TOK_LE, TOK_EQ, TOK_SELECT,
      TOK_MIN, TOK_MAX, TOK_NOT, TOK_LGAMMA, TOK_LOG1P, TOK_EXPM1, TOK_TAN, TOK_ATAN, TOK_TANH, TOK_FLOOR,
      TOK_RANDGAMMA, TOK_RANDPOISSON = Int32.(0:33)

function check(ctx, rc)
    rc == 0 && return nothing
    msg = unsafe_string(ccall((:ws_last_error, LIB), Cstring, (Ptr{Cvoid},), ctx))
    rc == -1 && throw(ArgumentError(msg))            # WS_EINVAL: the reference throws ArgumentError / error(...)
    rc == -5 && throw(UnsupportedModelError(msg))    # WS_EUNSUPPORTED
    error("wsb200 error $rc: $msg")
end

# ---- storage backend (src/stores.jl:28-35) -------------------------------------------------------------------------
mutable struct DeviceColumnStore <: AbstractParticleStore
    ctx::Ptr{Cvoid}
    n::Int
end

function DeviceColumnStore(n::Integer; device=0, seed=0, ess_perc_min=0.5, resampler=0)
    ref = Ref{Ptr{Cvoid}}(C_NULL)
    check(C_NULL, ccall((:ws_create, LIB), Cint, (Ref{Ptr{Cvoid}}, Int64, Cint, UInt64, Cdouble, Cint),
                        ref, n, device, seed, ess_perc_min, resampler))
    s = DeviceColumnStore(ref[], Int(n))
    finalizer(s -> ccall((:ws_destroy, LIB), Cint, (Ptr{Cvoid},), s.ctx), s)
    return s
end

"""
    DeviceSMCState(n; ess_perc_min = 0.5, seed = 0, device = 0, resampler = 0)

`SMCState` (src/types.jl:48-65) over a `DeviceColumnStore`.  The log-weights live in the library, so the host
`weights` field stays empty (the reference's convenience constructor would allocate `zeros(N)` on the host).
"""
function DeviceSMCState(n::Integer; ess_perc_min=0.5, seed=0, device=0, resampler=0, show_progress=false)
    store = DeviceColumnStore(n; device=device, seed=seed, ess_perc_min=ess_perc_min, resampler=resampler)
    st = SMCState(store; ess_perc_min=ess_perc_min, show_progress=show_progress)
    empty!(st.weights)
    return st
end
const DeviceState = SMCState{DeviceColumnStore}
ctx(state::DeviceState) = state.store.ctx

nparticles(s::DeviceColumnStore) = s.n

function lookup(s::DeviceColumnStore, name::Symbol)
    id = Ref{Int32}(-1); w = Ref{Int32}(0)
    check(s.ctx, ccall((:ws_col_lookup, LIB), Cint, (Ptr{Cvoid}, Cstring, Ref{Int32}, Ref{Int32}), s.ctx, String(name), id, w))
    return id[], w[]
end
function ensure(s::DeviceColumnStore, name::Symbol, width::Integer)
    id = Ref{Int32}(-1)
    check(s.ctx, ccall((:ws_col_ensure, LIB), Cint, (Ptr{Cvoid}, Cstring, Int32, Ref{Int32}), s.ctx, String(name), width, id))
    return id[]
end
hascol(s::DeviceColumnStore, name::Symbol) = lookup(s, name)[1] >= 0          # src/stores.jl:30

function colnames(s::DeviceColumnStore)
    cnt = Ref{Int32}(0)
    check(s.ctx, ccall((:ws_col_count, LIB), Cint, (Ptr{Cvoid}, Ref{Int32}), s.ctx, cnt))
    buf = Vector{UInt8}(undef, 256); w = Ref{Int32}(0)
    map(0:cnt[]-1) do i
        check(s.ctx, ccall((:ws_col_info, LIB), Cint, (Ptr{Cvoid}, Int32, Ptr{UInt8}, Int32, Ref{Int32}), s.ctx, i, buf, 256, w))
        Symbol(unsafe_string(pointer(buf)))
    end
end

# resample!(store, indices): particle i <- old particle indices[i] (1-based in Julia, 0-based in the ABI)
function resample!(s::DeviceColumnStore, indices::AbstractVector{<:Integer})
    idx = Int32.(indices .- 1)
    check(s.ctx, ccall((:ws_gather, LIB), Cint, (Ptr{Cvoid}, Ptr{Int32}), s.ctx, idx))
end

# ---- lazy per-particle values: what `vectorize` builds, as postfix tokens --------------------------------------------
"A per-particle scalar that lives on the device: a column plane or an expression over planes (postfix tokens)."
struct DeviceVec
    store::DeviceColumnStore
    toks::Vector{WsTok}
end
"A per-particle d-vector (the reference's `Vector{Vector{Float64}}` column): one `DeviceVec` per component."
struct DeviceVecN
    store::DeviceColumnStore
    comps::Vector{DeviceVec}
end
const Lazy = Union{DeviceVec,DeviceVecN}
tok(op, col=0, comp=0, val=0.0) = WsTok(Int32(op), Int32(col), Int32(comp), Int32(0), Float64(val))
constvec(s, c::Real) = DeviceVec(s, [tok(TOK_CONST, 0, 0, c)])
is_plane(v::DeviceVec) = length(v.toks) == 1 && v.toks[1].op == TOK_PLANE
cexpr(e::DeviceVec) = WsExpr(pointer(e.toks), length(e.toks), 0)

# getcol returns the lazy handle; `collect` / `Array` download a host copy (src/stores.jl:31)
function getcol(s::DeviceColumnStore, name::Symbol)
    id, w = lookup(s, name)
    id >= 0 || throw(KeyError(name))
    planes = [DeviceVec(s, [tok(TOK_PLANE, id, k - 1)]) for k in 1:w]
    return w == 1 ? planes[1] : DeviceVecN(s, planes)
end
Base.length(v::Lazy) = v.store.n
Base.size(v::Lazy) = (v.store.n,)
Base.axes(v::Lazy) = (Base.OneTo(v.store.n),)
Base.ndims(::Type{<:Lazy}) = 1
Base.eltype(::Type{DeviceVec}) = Float64
Base.eltype(::Type{DeviceVecN}) = Vector{Float64}
Base.broadcastable(v::Lazy) = v
function Base.collect(v::DeviceVec)
    is_plane(v) || error("only a stored column can be downloaded; assign the expression to a column first")
    out = Matrix{Float64}(undef, v.store.n, lookup_width(v))
    check(v.store.ctx, ccall((:ws_col_download, LIB), Cint, (Ptr{Cvoid}, Int32, Ptr{Float64}), v.store.ctx, v.toks[1].col, out))
    return out[:, v.toks[1].comp + 1]
end
Base.collect(v::DeviceVecN) = (cols = map(collect, v.comps); [[c[i] for c in cols] for i in 1:v.store.n])
Base.Array(v::Lazy) = collect(v)
function lookup_width(v::DeviceVec)
    w = Ref{Int32}(0); buf = Vector{UInt8}(undef, 256)
    check(v.store.ctx, ccall((:ws_col_info, LIB), Cint, (Ptr{Cvoid}, Int32, Ptr{UInt8}, Int32, Ref{Int32}), v.store.ctx, v.toks[1].col, buf, 256, w))
    return Int(w[])
end

# -- scalar-level algebra on lazies (used by `lower` and when a user helper function is traced) --
un(op, a::DeviceVec) = DeviceVec(a.store, vcat(a.toks, tok(op)))
bin(op, a::DeviceVec, b::DeviceVec) = DeviceVec(a.store, vcat(a.toks, b.toks, tok(op)))
bin(op, a::DeviceVec, b::Real) = bin(op, a, constvec(a.store, b))
bin(op, a::Real, b::DeviceVec) = bin(op, constvec(b.store, a), b)
for (f, op) in ((:+, TOK_ADD), (:-, TOK_SUB), (:*, TOK_MUL), (:/, TOK_DIV), (:^, TOK_POW), (:<, TOK_LT), (:<=, TOK_LE),
                (:(==), TOK_EQ), (:min, TOK_MIN), (:max, TOK_MAX))
    @eval Base.$f(a::DeviceVec, b::DeviceVec) = bin($op, a, b)
    @eval Base.$f(a::DeviceVec, b::Real) = bin($op, a, b)
    @eval Base.$f(a::Real, b::DeviceVec) = bin($op, a, b)
end
for (A, B) in ((:DeviceVec, :DeviceVec), (:DeviceVec, :Real), (:Real, :DeviceVec))
    @eval Base.:>(a::$A, b::$B) = b < a
    @eval Base.:>=(a::$A, b::$B) = b <= a
end
Base.:|(a::DeviceVec, b::DeviceVec) = bin(TOK_MAX, a, b)       # Bool columns are 1.0 / 0.0 planes: a || b
Base.:&(a::DeviceVec, b::DeviceVec) = bin(TOK_MIN, a, b)       # a && b
Base.:!(a::DeviceVec) = un(TOK_NOT, a)
Base.:-(a::DeviceVec) = un(TOK_NEG, a)
for (f, op) in ((:exp, TOK_EXP), (:log, TOK_LOG), (:sqrt, TOK_SQRT), (:sin, TOK_SIN), (:cos, TOK_COS), (:abs, TOK_ABS),
                (:abs2, TOK_SQUARE), (:log1p, TOK_LOG1P), (:expm1, TOK_EXPM1), (:tan, TOK_TAN), (:atan, TOK_ATAN),
                (:tanh, TOK_TANH), (:floor, TOK_FLOOR))
    @eval Base.$f(a::DeviceVec) = un($op, a)
end
loggamma(a::DeviceVec) = un(TOK_LGAMMA, a)
Base.ifelse(c::DeviceVec, a::Union{DeviceVec,Real}, b::Union{DeviceVec,Real}) =
    DeviceVec(c.store, vcat(c.toks, tovec(c.store, a).toks, tovec(c.store, b).toks, tok(TOK_SELECT)))
tovec(s, a::DeviceVec) = a
tovec(s, a::Real) = constvec(s, a)
Base.:+(a::DeviceVecN, b::DeviceVecN) = DeviceVecN(a.store, a.comps .+ b.comps)
Base.:-(a::DeviceVecN, b::DeviceVecN) = DeviceVecN(a.store, a.comps .- b.comps)
Base.:+(a::DeviceVecN, b::AbstractVector{<:Real}) = DeviceVecN(a.store, [a.comps[k] + b[k] for k in eachindex(b)])
Base.:+(a::AbstractVector{<:Real}, b::DeviceVecN) = b + a
Base.:-(a::DeviceVecN, b::AbstractVector{<:Real}) = DeviceVecN(a.store, [a.comps[k] - b[k] for k in eachindex(b)])
Base.:*(a::Real, b::DeviceVecN) = DeviceVecN(b.store, [a * c for c in b.comps])
Base.:*(a::DeviceVec, b::DeviceVecN) = DeviceVecN(b.store, [a * c for c in b.comps])
Base.:*(a::DeviceVecN, b::Union{Real,DeviceVec}) = b * a
Base.getindex(a::DeviceVecN, j::Integer) = a.comps[j]                      # `x[j]` on a vector column: plane j
# fresh variates inside a sampler expression (user kernels written for the device)
randn_tok(s) = DeviceVec(s, [tok(TOK_RANDN)]); randu_tok(s) = DeviceVec(s, [tok(TOK_RANDU)]); randexp_tok(s) = DeviceVec(s, [tok(TOK_RANDEXP)])
randgamma_tok(a::DeviceVec) = un(TOK_RANDGAMMA, a); randpoisson_tok(a::DeviceVec) = un(TOK_RANDPOISSON, a)

# -- the broadcast style: materialising a fused broadcast over lazies SERIALISES it --
struct DeviceStyle <: Broadcast.BroadcastStyle end
Base.BroadcastStyle(::Type{<:Lazy}) = DeviceStyle()
Base.BroadcastStyle(s::DeviceStyle, ::Broadcast.DefaultArrayStyle{0}) = s          # Ref(c) and scalars
Base.BroadcastStyle(s::DeviceStyle, ::Broadcast.AbstractArrayStyle) =
    unsupported("a host array inside a broadcast over device columns")
Base.BroadcastStyle(s::DeviceStyle, ::DeviceStyle) = s
Broadcast.instantiate(bc::Broadcast.Broadcasted{DeviceStyle}) = bc
Base.copy(bc::Broadcast.Broadcasted{DeviceStyle}) = lower(bc)
Base.copyto!(dest::Lazy, bc::Broadcast.Broadcasted{DeviceStyle}) = unsupported("in-place broadcast into a device column")

"the device store an expression is attached to"
storeof(x::Lazy) = x.store
storeof(x::Broadcast.Broadcasted) = (for a in x.args; s = storeof(a); s === nothing || return s; end; nothing)
storeof(x) = nothing

"`lower(x)`: Broadcasted tree -> DeviceVec / DeviceVecN / host constant (src/rewrites.jl:146-219 in reverse)"
lower(x::Lazy) = x
lower(x::Base.RefValue) = x[]
lower(x::Tuple{Any}) = x[1]
lower(x) = x
function lower(bc::Broadcast.Broadcasted)
    args = map(lower, bc.args)
    any(a -> a isa Lazy, args) || return bc.f(args...)                     # build-time constants fold on the host
    return call_lazy(bc.f, args...)
end
# `setindex!.(col, values, Ref(j))` — the write half of `x[j] .= rhs` / `x[j] ~ ...` (src/rewrites.jl: accessor_write_fn)
function call_lazy(::typeof(setindex!), target::DeviceVecN, value, j::Integer)
    s = target.store
    dst = target.comps[j].toks[1]
    rhs = tovec(s, value)
    GC.@preserve rhs check(s.ctx, ccall((:ws_assign, LIB), Cint, (Ptr{Cvoid}, Int32, Int32, Ref{WsExpr}), s.ctx, dst.col, dst.comp, cexpr(rhs)))
    return target
end
call_lazy(::typeof(getindex), a::DeviceVecN, j::Integer) = a.comps[j]
call_lazy(::typeof(identity), a) = a
call_lazy(::typeof(getproperty), a, p) = unsupported("struct-valued columns (`x.p`)")
# anything else: apply the function to the lazies themselves — the overloads above turn arithmetic, comparisons,
# `ifelse` and elementary functions into tokens, and a user helper `f(x) = a * exp(-x)` is traced the same way;
# `(xs...) -> [xs...]` (a vector literal of particle scalars) comes back as a Vector and becomes a DeviceVecN
function call_lazy(f, args...)
    r = try
        f(args...)
    catch err
        err isa UnsupportedModelError && rethrow()
        unsupported("function `$f` applied to particle variables ($(sprint(showerror, err)))")
    end
    r isa Lazy && return r
    if r isa AbstractVector
        s = something(map(storeof, args)...)
        return DeviceVecN(s, [tovec(s, c) for c in r])
    end
    r isa Real && return r
    unsupported("function `$f` returned a $(typeof(r)) for particle arguments")
end

# ---- the only write path: broadcast_setcol!(store, name, f, args) (src/stores.jl:33,85-96) -----------------------------
# Assign.apply! calls it with f = identity and the already-lowered right-hand side (src/transformers.jl:28-32), so the
# reference's own `apply!(::Assign)` runs unmodified.
function broadcast_setcol!(s::DeviceColumnStore, name::Symbol, ::typeof(identity), args::Tuple{Any})
    v = lower(args[1])
    if v isa DeviceVecN || v isa AbstractVector{<:Real}
        comps = v isa DeviceVecN ? v.comps : [constvec(s, c) for c in v]     # `θ .= zeros(J)`: one plane per component
        id = ensure(s, name, length(comps))
        GC.@preserve comps begin
            es = [cexpr(c) for c in comps]
            check(s.ctx, ccall((:ws_assign_vec, LIB), Cint, (Ptr{Cvoid}, Int32, Int32, Ptr{WsExpr}), s.ctx, id, length(comps), es))
        end
    elseif v isa DeviceVec || v isa Real
        rhs = tovec(s, v)
        id = ensure(s, name, 1)
        GC.@preserve rhs check(s.ctx, ccall((:ws_assign, LIB), Cint, (Ptr{Cvoid}, Int32, Int32, Ref{WsExpr}), s.ctx, id, 0, cexpr(rhs)))
    else
        unsupported("column $name of element type $(typeof(v))")
    end
    return nothing
end
broadcast_setcol!(::DeviceColumnStore, name::Symbol, f, args::Tuple) =
    unsupported("column $name: host closure `$f` cannot run on the device")

# ---- kernels: the reference's table entries, matched by identity -----------------------------------------------------
const DK = WeightedSampling.default_kernels
const NATIVE = IdDict{Any,Symbol}(DK.Normal => :Normal, DK.MvNormal => :MvNormal, DK.Exponential => :Exponential)
# kernels lowered to device expressions: (sampler(store, args...), logpdf(args..., x)); formulas as in
# weightedsampling.jl_b200/core.py `_expr_kernels` (Distributions.jl 0.25 `rand` / `logpdf`)
const EXPR_KERNELS = IdDict{Any,Tuple{Function,Function}}(
    DK.Uniform => ((s, a, b) -> a + (b - a) * randu_tok(s), (a, b, x) -> ifelse((x >= a) & (x <= b), -log(b - a), -Inf)),
    DK.LogNormal => ((s, m, sd) -> exp(m + sd * randn_tok(s)),
                     (m, sd, x) -> ifelse(x > 0.0, -(((log(x) - m) / sd)^2 + log(2pi)) / 2 - log(sd) - log(x), -Inf)),
    DK.Bernoulli => ((s, p) -> randu_tok(s) < p, (p, x) -> ifelse(x, log(p), log1p(-p))),
    DK.Laplace => ((s, m, t) -> m + t * (randexp_tok(s) - randexp_tok(s)), (m, t, x) -> -abs(x - m) / t - log(2.0 * t)),
    DK.Cauchy => ((s, m, t) -> m + t * tan(pi * (randu_tok(s) - 0.5)), (m, t, x) -> -log(pi) - log(t) - log1p(((x - m) / t)^2)),
    DK.Gamma => ((s, a, t) -> t * randgamma_tok(tovec(s, a)),
                 (a, t, x) -> ifelse(x >= 0.0, (a - 1.0) * log(x) - x / t - loggamma_any(a) - a * log(t), -Inf)),
    DK.Beta => ((s, a, b) -> 1.0 / (1.0 + randgamma_tok(tovec(s, b)) / randgamma_tok(tovec(s, a))),
                (a, b, x) -> ifelse((x >= 0.0) & (x <= 1.0), (a - 1.0) * log(x) + (b - 1.0) * log1p(-x) -
                                    (loggamma_any(a) + loggamma_any(b) - loggamma_any(a + b)), -Inf)),
    DK.TDist => ((s, v) -> randn_tok(s) / sqrt(2.0 * randgamma_tok(tovec(s, v / 2.0)) / v),
                 (v, x) -> loggamma_any((v + 1.0) / 2.0) - loggamma_any(v / 2.0) - 0.5 * log(v * pi) - (v + 1.0) / 2.0 * log1p(x * x / v)),
    DK.Chisq => ((s, v) -> 2.0 * randgamma_tok(tovec(s, v / 2.0)),
                 (v, x) -> ifelse(x >= 0.0, (v / 2.0 - 1.0) * log(x) - x / 2.0 - loggamma_any(v / 2.0) - (v / 2.0) * log(2.0), -Inf)),
    DK.InverseGamma => ((s, a, t) -> t / randgamma_tok(tovec(s, a)),
                        (a, t, x) -> ifelse(x > 0.0, a * log(t) - loggamma_any(a) - (a + 1.0) * log(x) - t / x, -Inf)),
    DK.Poisson => ((s, l) -> randpoisson_tok(tovec(s, l)), (l, x) -> ifelse(x >= 0.0, x * log(l) - l - loggamma_any(x + 1.0), -Inf)),
)
loggamma_any(a::DeviceVec) = loggamma(a)   # (every argument reaches these closures as a DeviceVec; constants are folded by the library)
const DEVICE_KERNEL_NAMES = Set{Symbol}([:Normal, :MvNormal, :Exponential, :Uniform, :LogNormal, :Bernoulli, :Laplace, :Cauchy,
                                        :Gamma, :Beta, :TDist, :Chisq, :InverseGamma, :Poisson])

scalar(s, a) = (v = lower(a); v isa DeviceVec ? v : v isa Real ? constvec(s, v) : unsupported("argument of type $(typeof(v)) where a scalar is needed"))
vector(s, a) = (v = lower(a); v isa DeviceVecN ? v.comps : v isa AbstractVector{<:Real} ? [constvec(s, c) for c in v] :
                                unsupported("argument of type $(typeof(v)) where a vector is needed"))
constmatrix(a) = (m = lower(a); m isa AbstractMatrix{<:Real} ? collect(vec(permutedims(Matrix{Float64}(m)))) :   # row-major for the ABI
                                unsupported("MvNormal covariance must be a build-time constant matrix"))

"target plane(s) of a Sample: `lhs::Symbol` (created on first write) or an accessor read `getindex.(col, Ref(j))`"
function target_plane(s::DeviceColumnStore, lhs::Symbol, width::Integer)
    return ensure(s, lhs, width), Int32(0)
end

# x ~ K(args...)                                                                 (src/transformers.jl:172-182)
function sample_into!(state::DeviceState, kernel, col::Int32, comp::Int32, args::Tuple, vector_width::Integer=0)
    s = state.store
    name = get(NATIVE, kernel, nothing)
    if name === :Normal
        mu, sg = scalar(s, args[1]), scalar(s, args[2])
        GC.@preserve mu sg check(s.ctx, ccall((:ws_sample_normal, LIB), Cint, (Ptr{Cvoid}, Int32, Int32, Ref{WsExpr}, Ref{WsExpr}),
                                              s.ctx, col, comp, cexpr(mu), cexpr(sg)))
    elseif name === :Exponential
        th = scalar(s, args[1])
        GC.@preserve th check(s.ctx, ccall((:ws_sample_exponential, LIB), Cint, (Ptr{Cvoid}, Int32, Int32, Ref{WsExpr}), s.ctx, col, comp, cexpr(th)))
    elseif name === :MvNormal
        mu = vector(s, args[1]); cov = constmatrix(args[2])
        GC.@preserve mu begin
            es = [cexpr(c) for c in mu]
            check(s.ctx, ccall((:ws_sample_mvnormal, LIB), Cint, (Ptr{Cvoid}, Int32, Int32, Ptr{WsExpr}, Ptr{Float64}), s.ctx, col, length(mu), es, cov))
        end
    else
        pair = get(EXPR_KERNELS, kernel, nothing)
        pair === nothing && unsupported("kernel $(kernel_label(kernel))")
        largs = map(a -> scalar(s, a), args)
        x = DeviceVec(s, [tok(TOK_PLANE, col, comp)])
        smp = tovec(s, pair[1](s, largs...))
        lpd = tovec(s, pair[2](largs..., x))
        GC.@preserve smp lpd check(s.ctx, ccall((:ws_sample_expr, LIB), Cint, (Ptr{Cvoid}, Int32, Int32, Ref{WsExpr}, Ptr{WsExpr}, Ref{WsExpr}),
                                                s.ctx, col, comp, cexpr(smp), C_NULL, cexpr(lpd)))
    end
    return nothing
end
kernel_label(k) = (for (name, v) in pairs(DK); v === k && return String(name); end; "a user WeightedKernel (host closures)")

function apply!(t::Sample, state::DeviceState)
    args = t.argfn(state)
    s = state.store
    width = get(NATIVE, t.kernel, nothing) === :MvNormal ? length(vector(s, args[1])) : 1
    col = ensure(s, t.lhs, width)
    sample_into!(state, t.kernel, col, Int32(0), args)
    advance!(state)
    return nothing
end
# x[j] ~ K(args...): the accessor's read closure names the plane                    (src/transformers.jl:118-131)
function apply!(t::AccessorSample, state::DeviceState)
    args = t.argfn(state)
    dst = lower(t.readfn(state))
    dst isa DeviceVec && is_plane(dst) || unsupported("accessor sampling target that is not one plane of a vector column")
    sample_into!(state, t.kernel, dst.toks[1].col, dst.toks[1].comp, args)
    advance!(state)
    return nothing
end
# expr => K(args...)                                                                 (src/transformers.jl:228-235)
function observe!(state::DeviceState, kernel, obs, args::Tuple)
    s = state.store
    name = get(NATIVE, kernel, nothing)
    if name === :Normal
        o, mu, sg = scalar(s, obs), scalar(s, args[1]), scalar(s, args[2])
        GC.@preserve o mu sg check(s.ctx, ccall((:ws_observe_normal, LIB), Cint, (Ptr{Cvoid}, Ref{WsExpr}, Ref{WsExpr}, Ref{WsExpr}),
                                                s.ctx, cexpr(o), cexpr(mu), cexpr(sg)))
    elseif name === :Exponential
        o, th = scalar(s, obs), scalar(s, args[1])
        GC.@preserve o th check(s.ctx, ccall((:ws_observe_exponential, LIB), Cint, (Ptr{Cvoid}, Ref{WsExpr}, Ref{WsExpr}), s.ctx, cexpr(o), cexpr(th)))
    elseif name === :MvNormal
        o, mu = vector(s, obs), vector(s, args[1]); cov = constmatrix(args[2])
        GC.@preserve o mu begin
            eo = [cexpr(c) for c in o]; em = [cexpr(c) for c in mu]
            check(s.ctx, ccall((:ws_observe_mvnormal, LIB), Cint, (Ptr{Cvoid}, Int32, Ptr{WsExpr}, Ptr{WsExpr}, Ptr{Float64}),
                               s.ctx, length(mu), eo, em, cov))
        end
    else
        pair = get(EXPR_KERNELS, kernel, nothing)
        pair === nothing && unsupported("kernel $(kernel_label(kernel))")
        term = tovec(s, pair[2](map(a -> scalar(s, a), args)..., scalar(s, obs)))
        GC.@preserve term check(s.ctx, ccall((:ws_weight_expr, LIB), Cint, (Ptr{Cvoid}, Ref{WsExpr}), s.ctx, cexpr(term)))
    end
    state.weights_changed = true
    return nothing
end
function apply!(t::Observe, state::DeviceState)
    observe!(state, t.kernel, t.lhsfn(state), t.argfn(state))
    advance!(state)
    return nothing
end
# _ ~ K(args..., x): a Weight's kernel takes the value as its last argument          (src/transformers.jl:283-289)
function apply!(t::Weight, state::DeviceState)
    args = t.argfn(state)
    observe!(state, t.kernel, args[end], args[1:end-1])
    advance!(state)
    return nothing
end

# Resample.apply! — the whole state machine runs inside ws_resample              (src/transformers.jl:474-498)
function apply!(::Resample, state::DeviceState)
    info = Ref(WsResampleInfo())
    check(ctx(state), ccall((:ws_resample, LIB), Cint, (Ptr{Cvoid}, Ref{WsResampleInfo}), ctx(state), info))
    if info[].fired != 0
        state.resampled = info[].resampled != 0
        state.weights_changed = false
    end
    return nothing
end

# Move.apply! with the reference's proposals, matched by identity               (src/transformers.jl:588-623)
function apply!(t::Move, state::DeviceState)
    s = state.store
    proposal = t.proposal === WeightedSampling.RW ? Int32(0) : t.proposal === WeightedSampling.autoRW ? Int32(1) :
               unsupported("proposal `$(t.proposal)` (host closure)")
    args = t.argfn(state)
    cols = Int32[]; comps = Int32[]
    for c in t.targets
        id, w = lookup(s, c)
        id >= 0 || throw(KeyError(c))
        for k in 0:w-1
            push!(cols, id); push!(comps, k)
        end
    end
    d = length(cols)
    step = length(args) >= 1 ? Float64(first(args[1])) : (proposal == 0 ? error("RW needs a step size") : 1e-3)
    bounds = length(args) >= 2 ? args[2] : nothing
    lo = Float64[]; hi = Float64[]
    if bounds !== nothing
        bl = bounds isa Tuple{<:Real,<:Real} ? fill(bounds, d) : collect(bounds)       # src/move_kernels.jl:23-28
        length(bl) == d || throw(ArgumentError("bounds must have length $d (one (lo, hi) tuple per target)"))
        lo = Float64[b[1] for b in bl]; hi = Float64[b[2] for b in bl]
    end
    div = t.diversity_threshold === nothing ? NaN : Float64(t.diversity_threshold)
    info = Ref(WsMoveInfo(0, 0, NaN, 0))
    GC.@preserve cols comps lo hi begin
        spec = WsMoveSpec(d, pointer(cols), pointer(comps), proposal, isempty(lo) ? 0 : 1,
                          isempty(lo) ? C_NULL : pointer(lo), isempty(hi) ? C_NULL : pointer(hi), step, div, -1)
        check(ctx(state), ccall((:ws_move, LIB), Cint, (Ptr{Cvoid}, Ref{WsMoveSpec}, Ref{WsMoveInfo}), ctx(state), spec, info))
    end
    return nothing                                  # depth-neutral, weights untouched
end

# run!: the library keeps its own depth counter and score tape                    (src/types.jl:120-126)
function run!(root::ParticleTransformer, state::DeviceState)
    check(ctx(state), ccall((:ws_begin_run, LIB), Cint, (Ptr{Cvoid},), ctx(state)))
    state.root = root
    state.depth = 0
    apply!(root, state)
    return state
end

# score!: the library records the tape as the statements execute and ws_move folds it on the device; on the host
# the walk only has to keep the depth counter in step (so that a user-level `score_logpdf` cut-off means the same).
score!(::Union{Sample,AccessorSample,Observe,Weight}, ::DeviceState, c::ScoreCtx) = (advance!(c); nothing)
function score_logpdf(state::DeviceState, targets, target_depth::Int)              # src/types.jl:183-206
    out = Vector{Float64}(undef, state.store.n)
    check(ctx(state), ccall((:ws_score_logpdf, LIB), Cint, (Ptr{Cvoid}, Int64, Ptr{Float64}), ctx(state), target_depth, out))
    return out
end

# ---- @device_model: `@model` + the device-op check at macro-expansion time -------------------------------------------
"kernel names used by `~` / `=>` statements anywhere in a model body"
function kernel_names!(acc::Vector{Symbol}, ex)
    if ex isa Expr
        if ex.head == :call && length(ex.args) == 3 && ex.args[1] in (:~, :(=>)) && ex.args[3] isa Expr &&
           ex.args[3].head == :call && ex.args[3].args[1] isa Symbol
            push!(acc, ex.args[3].args[1])
        end
        foreach(a -> kernel_names!(acc, a), ex.args)
    end
    return acc
end
"""
    WSB200.@device_model function name(args...) ... end

The reference's `@model` (src/rewrites.jl:787-806) with one extra check: a statement whose kernel is one of the
reference's `default_kernels` but has no device lowering (`Wishart`, `Dirichlet`, `LKJ`, ...) is an error at MACRO
EXPANSION, not at run time.  Names that are not table entries (user kernels passed through `kernels = (...)`) are
checked when the statement first executes.
"""
macro device_model(ex)
    for k in kernel_names!(Symbol[], ex)
        if hasproperty(DK, k) && !(k in DEVICE_KERNEL_NAMES)
            error("@device_model: kernel `$k` is in WeightedSampling.default_kernels but outside the device-op set of libwsb200 " *
                  "(supported: $(join(sort(collect(DEVICE_KERNEL_NAMES)), ", ")))")
        end
    end
    return esc(:(WeightedSampling.@model $ex))
end

# ---- analysis (src/utils.jl) -------------------------------------------------------------------------------------
function log_evidence(state::DeviceState)                                             # utils.jl:21
    le = Ref(0.0); ess = Ref(0.0)
    check(ctx(state), ccall((:ws_log_evidence, LIB), Cint, (Ptr{Cvoid}, Ref{Float64}, Ref{Float64}), ctx(state), le, ess))
    le[]
end
function exp_norm(state::DeviceState)                                                 # resampling.jl:72-77 on state.weights
    out = Vector{Float64}(undef, state.store.n)
    check(ctx(state), ccall((:ws_exp_norm, LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}), ctx(state), out))
    out
end
function weights(state::DeviceState)
    out = Vector{Float64}(undef, state.store.n)
    check(ctx(state), ccall((:ws_weights_download, LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}), ctx(state), out))
    out
end
"`@E(f, state)` (utils.jl:45-68) as a function: the argument NAMES of `f` are particle-variable names"
function expectation(f::Function, state::DeviceState)
    names = Base.method_argnames(first(methods(f)))[2:end]
    val = tovec(state.store, f((getcol(state.store, n) for n in names)...))
    out = Ref(0.0)
    GC.@preserve val begin
        e = Ref(cexpr(val))
        check(ctx(state), ccall((:ws_expectation, LIB), Cint, (Ptr{Cvoid}, Ref{WsExpr}, Int32, Ref{Float64}), ctx(state), e, 1, out))
    end
    out[]
end
# describe(state) (utils.jl:183-289): every statistic, including the StatsBase weighted median, on the device
function describe_plane(state::DeviceState, name::Symbol, comp::Integer=0)
    id, _ = lookup(state.store, name)
    out = Ref(WsPlaneStats(0, 0, 0, 0, 0, ntuple(_ -> 0.0, 8))); ess = Ref(0.0)
    check(ctx(state), ccall((:ws_describe, LIB), Cint, (Ptr{Cvoid}, Int32, Ref{Int32}, Ref{Int32}, Ref{WsPlaneStats}, Ref{Float64}),
                            ctx(state), 1, Ref(Int32(id)), Ref(Int32(comp)), out, ess))
    out[], ess[]
end
"""`sample(state, n; replace)` (utils.jl:102-118): 1-based GLOBAL particle indices and the rows of one column, drawn on
the device.  Collective on a sharded state: every rank calls it and gets the same indices and rows.
(Not executed in this repository's test suite: there is no Julia toolchain here.)"""
function sample_rows(state::DeviceState, name::Symbol, n::Integer; replace::Bool=true)
    idx = Vector{Int64}(undef, n)
    check(ctx(state), ccall((:ws_sample_indices, LIB), Cint, (Ptr{Cvoid}, Int64, Cint, Ptr{Int64}), ctx(state), n, replace, idx))
    id, w = lookup(state.store, name)
    rows = Matrix{Float64}(undef, n, w)
    check(ctx(state), ccall((:ws_col_download_global_rows, LIB), Cint, (Ptr{Cvoid}, Int32, Ptr{Int64}, Int64, Ptr{Float64}),
                            ctx(state), id, idx, n, rows))
    idx .+ 1, rows
end
function marginal_diversity(state::DeviceState, targets::Vector{Symbol})               # transformers.jl:560-565
    cols = Int32[]; comps = Int32[]
    for c in targets
        id, w = lookup(state.store, c)
        for k in 0:w-1; push!(cols, id); push!(comps, k); end
    end
    out = Ref(0.0)
    check(ctx(state), ccall((:ws_marginal_diversity, LIB), Cint, (Ptr{Cvoid}, Int32, Ptr{Int32}, Ptr{Int32}, Ref{Float64}),
                            ctx(state), length(cols), cols, comps, out))
    out[]
end
set_genealogy!(state::DeviceState, on::Bool; budget_bytes::Integer=0) =
    check(ctx(state), ccall((:ws_set_genealogy, LIB), Cint, (Ptr{Cvoid}, Cint, Int64), ctx(state), on, budget_bytes))

# ---- replayed standard variates (parity tests: SURVEY §8c consumption order) ---------------------------------------------
for (fn, sym) in ((:set_replay_normals, :ws_set_replay_normals), (:set_replay_uniforms, :ws_set_replay_uniforms),
                  (:set_replay_exponentials, :ws_set_replay_exponentials), (:set_replay_variates, :ws_set_replay_variates))
    @eval $fn(state::DeviceState, v::Vector{Float64}) =
        check(ctx(state), ccall(($(QuoteNode(sym)), LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}, Int64), ctx(state), v, length(v)))
end

# ---- one filter over several GPUs: one Julia process per GPU (INTEGRATION.md) ----------------------------------------
nccl_unique_id() = (buf = zeros(UInt8, 128); check(C_NULL, ccall((:ws_nccl_unique_id, LIB), Cint, (Ptr{UInt8},), buf)); buf)
function ShardedColumnStore(n_global::Integer, rank::Integer, nranks::Integer, id::Vector{UInt8}; device=rank, seed=0,
                            ess_perc_min=0.5, resampler=0)
    ref = Ref{Ptr{Cvoid}}(C_NULL)
    check(C_NULL, ccall((:ws_create_sharded, LIB), Cint, (Ref{Ptr{Cvoid}}, Int64, Cint, Cint, Ptr{UInt8}, Cint, UInt64, Cdouble, Cint),
                        ref, n_global, rank, nranks, id, device, seed, ess_perc_min, resampler))
    nl = Ref{Int64}(0); ng = Ref{Int64}(0)
    check(ref[], ccall((:ws_n_particles, LIB), Cint, (Ptr{Cvoid}, Ref{Int64}, Ref{Int64}), ref[], nl, ng))
    s = DeviceColumnStore(ref[], Int(nl[]))          # the rank's shard: global slots [rank N / R, (rank + 1) N / R)
    finalizer(s -> ccall((:ws_destroy, LIB), Cint, (Ptr{Cvoid},), s.ctx), s)
    return s
end

end # module
