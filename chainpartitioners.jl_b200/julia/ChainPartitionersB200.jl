# ChainPartitionersB200.jl -- the Julia-side binding a ChainPartitioners.jl maintainer would add
# (one more glue file next to src/glue_*.jl, or a same-named package): it keeps the reference's API
#   partition_stripe(A, K, method, args...; kwargs...)      (src/DynamicSplitter.jl:15,
#                                                            src/BisectCostBottleneckSplitter.jl:6,
#                                                            src/LazyBisectCostBottleneckSplitter.jl:8,140,260)
#   pack_stripe(A, method, args...; kwargs...)              (src/DynamicChunker.jl:20, src/ConvexTotalChunker.jl:141,
#                                                            src/OverlapChunker.jl:6, src/StrictChunker.jl:5)
#   oracle_stripe / bound_stripe                            (src/Costs.jl:3-19)
# and forwards to libchainb200.so (include/chainb200.h) with `ccall`.  Julia is not installed in the
# build image, so this file is NOT executed by the test-suite; it is deliberately mechanical: marshal
# colptr/rowval/coefficients, wrap the returned split vector in SplitPartition.  The Python mirror in
# chainpartitioners.jl_b200/api.py exercises exactly the same C entry points and is what the tests run.
module ChainPartitionersB200

using SparseArrays
using ChainPartitioners
import ChainPartitioners: partition_stripe, pack_stripe, partition_plaid, oracle_stripe, bound_stripe, bottleneck_value, total_value, adjointpattern,
    netcount, dianetcount, selfnetcount, selfpincount, pincount, dominancecount, dominancesum, rookcount!, rooksum!,
    AlternatingPartitioner, SymmetricPartitioner, DisjointPartitioner, MapPartition, DomainPartition,
    ConcaveTotalChunker, ConcaveTotalSplitter,
    AffineWorkModel, AffineConnectivityModel, AffineMonotonizedSymmetricConnectivityModel,
    AffineSymmetricConnectivityModel, AffineHyperedgeCutModel, AffineSymmetricEdgeCutModel, AffineEnvelopeModel,
    AffinePrimaryConnectivityModel, AffineSecondaryConnectivityModel, AffinePrimaryEdgeCutModel, AffineSecondaryEdgeCutModel,
    ColumnBlockComponentCostModel, BlockComponentCostModel, block_component,
    ConstrainedCost, VertexCount, FeasibleCost, SplitPartition,
    DynamicBottleneckSplitter, DynamicTotalSplitter, BisectCostBottleneckSplitter, BisectIndexBottleneckSplitter, LazyBisectCostBottleneckSplitter,
    FlipBisectCostBottleneckSplitter, LazyFlipBisectCostBottleneckSplitter, FlipBisectIndexBottleneckSplitter,
    DynamicBottleneckChunker, DynamicTotalChunker, ConvexTotalChunker, ConvexTotalSplitter, OverlapChunker, StrictChunker, EquiChunker, EquiSplitter

const lib = get(ENV, "CHAINB200_LIB", "libchainb200.so")

# The dispatch tag: wraps a method (partition_stripe(A, K, OnB200(DynamicBottleneckSplitter(f)))), a model
# (bottleneck_value(A, Φ, OnB200(f))) or a hint (oracle_stripe(OnB200(SparseHint()), f, A), netcount(OnB200(nothing), A)).
struct OnB200{Mtd}
    mtd::Mtd
end

# ---- C structs (binary layout of cpb_model / cpb_constraint) ---------------------------------
struct CModel
    kind::Int32
    is_float::Int32
    coef::NTuple{8, Float64}
    R::Int32
    w_tab::Int32
    u_tab::Int32
    _pad::Int32
    alpha_col::Ptr{Float64}
    beta_col::Ptr{Float64}
    beta_row::Ptr{Float64}
end

struct CConstraint
    enabled::Int32
    _pad::Int32
    w_coef::NTuple{3, Int64}
    w_max::Int64
end

struct CpbError <: Exception
    code::Int
    msg::String
end

check(rc) = rc == 0 ? nothing : throw(CpbError(rc, unsafe_string(ccall((:cpb_last_error, lib), Cstring, ()))))

pad8(xs...) = ntuple(i -> i <= length(xs) ? Float64(xs[i]) : 0.0, 8)
isfloat(::Type{<:AbstractFloat}) = Int32(1)
isfloat(::Type) = Int32(0)
affine(kind, ::Type{Tv}, xs...) where {Tv} = (CModel(kind, isfloat(Tv), pad8(xs...), 0, 0, 0, 0, C_NULL, C_NULL, C_NULL), Any[])

cmodel(m::AffineWorkModel{Tv}, args...) where {Tv} = affine(0, Tv, m.α, m.β_vertex, m.β_pin)
cmodel(m::AffineConnectivityModel{Tv}, args...) where {Tv} = affine(1, Tv, m.α, m.β_vertex, m.β_pin, m.β_net)
cmodel(m::AffineMonotonizedSymmetricConnectivityModel{Tv}, args...) where {Tv} = affine(2, Tv, m.α, m.β_vertex, m.β_over_pin, m.β_dia_net, m.Δ_pins)
cmodel(m::AffineSymmetricConnectivityModel{Tv}, args...) where {Tv} = affine(3, Tv, m.α, m.β_vertex, m.β_pin, m.β_local_net, m.β_remote_net)
cmodel(m::AffineHyperedgeCutModel{Tv}, args...) where {Tv} = affine(4, Tv, m.α, m.β_vertex, m.β_pin, m.β_self_net, m.β_cut_net)
cmodel(m::AffineSymmetricEdgeCutModel{Tv}, args...) where {Tv} = affine(5, Tv, m.α, m.β_vertex, m.β_self_pin, m.β_cut_pin)
cmodel(m::AffineEnvelopeModel{Tv}, args...) where {Tv} = affine(6, Tv, m.α, m.β_vertex, m.β_pin, m.β_net)
cmodel(m::AffinePrimaryConnectivityModel{Tv}, args...) where {Tv} = affine(9, Tv, m.α, m.β_vertex, m.β_pin, m.β_local_net, m.β_remote_net)  # needs Π
cmodel(m::AffineSecondaryConnectivityModel{Tv}, args...) where {Tv} = affine(10, Tv, m.α, m.β_vertex, m.β_pin, m.β_local_net, m.β_remote_net)  # needs Π
cmodel(m::AffinePrimaryEdgeCutModel{Tv}, args...) where {Tv} = affine(11, Tv, m.α, m.β_vertex, m.β_self_pin, m.β_cut_pin)  # needs Π
cmodel(m::AffineSecondaryEdgeCutModel{Tv}, args...) where {Tv} = affine(12, Tv, m.α, m.β_vertex, m.β_self_pin, m.β_cut_pin)  # needs Π

# Functors cannot cross the ABI: tabulate block_component(f, w) (src/BlockCosts.jl:41-44) for w = 0..w_tab
tab(f, hi) = Float64[w == 0 && !(f isa Function || f isa Number) ? 0.0 : block_component(f, w) for w in 0:hi]
function cmodel(m::ColumnBlockComponentCostModel{Tv}, w_tab, u_tab) where {Tv}
    a, b = tab(m.α_col, w_tab), tab(m.β_col, w_tab)
    (CModel(7, isfloat(Tv), pad8(), 1, w_tab, 0, 0, pointer(a), pointer(b), C_NULL), Any[a, b])
end
function cmodel(m::BlockComponentCostModel{Tv, R}, w_tab, u_tab) where {Tv, R}
    a = tab(m.α_col, w_tab)
    bc = reduce(vcat, (tab(f, w_tab) for f in m.β_col); init = Float64[])
    br = reduce(vcat, (tab(f, u_tab) for f in m.β_row); init = Float64[])
    (CModel(8, isfloat(Tv), pad8(), R, w_tab, u_tab, 0, pointer(a), pointer(bc), pointer(br)), Any[a, bc, br])
end

# ConstrainedCost(f, w, w_max) with a count weight (src/Costs.jl:105-147): w gets an oracle of its own on the same resident
# matrix and the solve goes through cpb_partition_stripe_weighted (Dynamic, Convex and Concave splitters)
const CountWeighted = Union{ConstrainedCost{<:Any, <:AffineConnectivityModel{<:Integer}},
                            ConstrainedCost{<:Any, <:AffineMonotonizedSymmetricConnectivityModel{<:Integer}}}

constraint(::Any) = CConstraint(0, 0, (0, 0, 0), 0)
constraint(c::ConstrainedCost{<:Any, VertexCount}) = CConstraint(1, 0, (0, 1, 0), Int64(c.w_max))
constraint(c::ConstrainedCost{<:Any, <:AffineWorkModel{<:Integer}}) = CConstraint(1, 0, (Int64(c.w.α), Int64(c.w.β_vertex), Int64(c.w.β_pin)), Int64(c.w_max))
constraint(c::ConstrainedCost{<:Any, FeasibleCost}) = CConstraint(0, 0, (0, 0, 0), 0)
# count weights (AffineConnectivityModel / AffineMonotonizedSymmetricConnectivityModel) cannot be expressed here: stripe_solve
# hands them to cpb_partition_stripe_weighted; pack_stripe has no count-weight form
constraint(c::CountWeighted) = throw(ArgumentError("pack_stripe takes VertexCount() or an integer AffineWorkModel weight; count weights are not built for the chunkers"))
basecost(f) = f
basecost(c::ConstrainedCost) = c.f

# ---- handles ---------------------------------------------------------------------------------
mutable struct DeviceMatrix
    h::Ptr{Cvoid}
    m::Int
    n::Int
    function DeviceMatrix(A::SparseMatrixCSC{Tv, Int64}) where {Tv}
        h = Ref{Ptr{Cvoid}}(C_NULL)
        (m, n) = size(A)
        GC.@preserve A check(ccall((:cpb_matrix_create, lib), Cint,
            (Int64, Int64, Int64, Ptr{Int64}, Ptr{Int64}, Ref{Ptr{Cvoid}}), m, n, nnz(A), A.colptr, A.rowval, h))
        finalizer(x -> ccall((:cpb_matrix_destroy, lib), Cvoid, (Ptr{Cvoid},), x.h), new(h[], m, n))
    end
    function DeviceMatrix(A::SparseMatrixCSC{Tv, Int32}) where {Tv}  # half the upload
        h = Ref{Ptr{Cvoid}}(C_NULL)
        (m, n) = size(A)
        GC.@preserve A check(ccall((:cpb_matrix_create_i32, lib), Cint,
            (Int64, Int64, Int64, Ptr{Int32}, Ptr{Int32}, Ref{Ptr{Cvoid}}), m, n, nnz(A), A.colptr, A.rowval, h))
        finalizer(x -> ccall((:cpb_matrix_destroy, lib), Cvoid, (Ptr{Cvoid},), x.h), new(h[], m, n))
    end
    DeviceMatrix(h::Ptr{Cvoid}, m::Int, n::Int) = finalizer(x -> ccall((:cpb_matrix_destroy, lib), Cvoid, (Ptr{Cvoid},), x.h), new(h, m, n))
end

# a handle the library made (cpb_adjointpattern, cpb_matrix_permute): same finalizer
function DeviceMatrix(h::Ptr{Cvoid})
    m, n, nz = Ref{Int64}(0), Ref{Int64}(0), Ref{Int64}(0)
    check(ccall((:cpb_matrix_dims, lib), Cint, (Ptr{Cvoid}, Ref{Int64}, Ref{Int64}, Ref{Int64}), h, m, n, nz))
    return DeviceMatrix(h, Int(m[]), Int(n[]))
end
Base.size(dA::DeviceMatrix) = (dA.m, dA.n)
device_matrix(A::DeviceMatrix) = A
device_matrix(A::SparseMatrixCSC) = DeviceMatrix(A)

# adjointpattern(A) on the device (src/util.jl:67-95): the transpose pattern stays in HBM
function adjointpattern(dA::DeviceMatrix)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:cpb_adjointpattern, lib), Cint, (Ptr{Cvoid}, Ref{Ptr{Cvoid}}), dA.h, h))
    return DeviceMatrix(h[])
end
# back to the host as a pattern matrix (cpb_matrix_get)
function SparseArrays.SparseMatrixCSC(dA::DeviceMatrix)
    m, n, nz = Ref{Int64}(0), Ref{Int64}(0), Ref{Int64}(0)
    check(ccall((:cpb_matrix_dims, lib), Cint, (Ptr{Cvoid}, Ref{Int64}, Ref{Int64}, Ref{Int64}), dA.h, m, n, nz))
    colptr, rowval = Vector{Int64}(undef, n[] + 1), Vector{Int64}(undef, nz[])
    check(ccall((:cpb_matrix_get, lib), Cint, (Ptr{Cvoid}, Ptr{Int64}, Ptr{Int64}), dA.h, colptr, rowval))
    return SparseMatrixCSC(Int(m[]), Int(n[]), colptr, rowval, ones(Bool, nz[]))
end

mutable struct DeviceOracle
    h::Ptr{Cvoid}
    A::DeviceMatrix
    function DeviceOracle(A::DeviceMatrix, f, Π = nothing; w_tab = A.n)
        u_tab = Π === nothing ? 0 : maximum(diff(Π.spl))
        (cm, keep) = cmodel(basecost(f), w_tab, u_tab)
        h = Ref{Ptr{Cvoid}}(C_NULL)
        spl = Π === nothing ? C_NULL : pointer(Π.spl)
        K = Π === nothing ? 0 : Π.K
        GC.@preserve keep Π check(ccall((:cpb_oracle_create, lib), Cint,
            (Ptr{Cvoid}, Ref{CModel}, Ptr{Int64}, Int64, Ref{Ptr{Cvoid}}), A.h, cm, spl, K, h))
        finalizer(x -> ccall((:cpb_oracle_destroy, lib), Cvoid, (Ptr{Cvoid},), x.h), new(h[], A))
    end
end

# ocl(j, j′[, k]) -- src/ConnectivityCosts.jl:58-64 and friends
function (ocl::DeviceOracle)(j::Integer, j′::Integer, k...)
    out = Ref{Float64}(0.0)
    check(ccall((:cpb_oracle_query, lib), Cint, (Ptr{Cvoid}, Int64, Ref{Int64}, Ref{Int64}, Ptr{Int64}, Ref{Float64}),
                ocl.h, 1, Int64(j), Int64(j′), C_NULL, out))
    return out[]
end
function query(ocl::DeviceOracle, j::Vector{Int64}, j′::Vector{Int64})
    out = Vector{Float64}(undef, length(j))
    check(ccall((:cpb_oracle_query, lib), Cint, (Ptr{Cvoid}, Int64, Ptr{Int64}, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}),
                ocl.h, length(j), j, j′, C_NULL, out))
    return out
end

# ocl(j, j′, k) for the row-partition-aware models (PrimaryConnectivityCosts.jl:66-73, ...): k = part index
function (ocl::DeviceOracle)(j::Integer, j′::Integer, k::Integer)
    out = Ref{Float64}(0.0)
    check(ccall((:cpb_oracle_query, lib), Cint, (Ptr{Cvoid}, Int64, Ref{Int64}, Ref{Int64}, Ref{Int64}, Ref{Float64}),
                ocl.h, 1, Int64(j), Int64(j′), Int64(k), out))
    return out[]
end

# oracle_stripe(OnB200(hint), mdl, A[, Π]) (src/Costs.jl:3-7): the wrapper takes the place of the hint; A may be a
# SparseMatrixCSC (uploaded once, kept alive by the oracle) or a DeviceMatrix
oracle_stripe(::OnB200, mdl, A, args...; kwargs...) = DeviceOracle(device_matrix(A), mdl, args...)

# bottleneck_value / total_value (src/Costs.jl:26-66) of a SplitPartition; Map- and DomainPartitions are first made
# contiguous by gathering the columns part by part on the device (cpb_matrix_permute), as compute_objective does with
# A[:, Φ_dom.prm]
function objective(total::Bool, A, Φ::SplitPartition, f::OnB200, Π...)
    ocl = DeviceOracle(device_matrix(A), f.mtd, Π...)
    out = Ref{Float64}(0.0)
    spl = Vector{Int64}(Φ.spl)
    check(ccall((:cpb_objective, lib), Cint, (Ptr{Cvoid}, Cint, Int64, Ptr{Int64}, Ref{Float64}), ocl.h, total ? 1 : 0, Φ.K, spl, out))
    return out[]
end
function objective(total::Bool, A, Φ::Union{MapPartition, DomainPartition}, f::OnB200, Π...)
    Φ_dom = convert(DomainPartition, Φ)
    dA = device_matrix(A)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    prm = Vector{Int64}(Φ_dom.prm)
    check(ccall((:cpb_matrix_permute, lib), Cint, (Ptr{Cvoid}, Ptr{Int64}, Ptr{Int64}, Ref{Ptr{Cvoid}}), dA.h, prm, C_NULL, h))
    return objective(total, DeviceMatrix(h[]), SplitPartition{Int64}(Φ_dom.K, Vector{Int64}(Φ_dom.spl)), f, Π...)
end
bottleneck_value(A, Φ, f::OnB200, Π...) = objective(false, A, Φ, f, Π...)
total_value(A, Φ, f::OnB200, Π...) = objective(true, A, Φ, f, Π...)

# colour arrays (src/SparseColorArrays.jl): netcount(OnB200(hint), A)[j, j′] etc. through cpb_count_query
struct DeviceColorArray
    which::Cint
    A::DeviceMatrix
end
function Base.getindex(c::DeviceColorArray, j::Integer, j′::Integer)
    out = Ref{Int64}(0)
    check(ccall((:cpb_count_query, lib), Cint, (Ptr{Cvoid}, Cint, Int64, Ref{Int64}, Ref{Int64}, Ref{Int64}), c.A.h, c.which, 1, Int64(j), Int64(j′), out))
    return out[]
end
function query(c::DeviceColorArray, j::Vector{Int64}, j′::Vector{Int64})
    out = Vector{Int64}(undef, length(j))
    check(ccall((:cpb_count_query, lib), Cint, (Ptr{Cvoid}, Cint, Int64, Ptr{Int64}, Ptr{Int64}, Ptr{Int64}), c.A.h, c.which, length(j), j, j′, out))
    return out
end
pincount(::OnB200, A; kwargs...) = DeviceColorArray(0, device_matrix(A))
netcount(::OnB200, A; kwargs...) = DeviceColorArray(1, device_matrix(A))
dianetcount(::OnB200, A; kwargs...) = DeviceColorArray(2, device_matrix(A))
selfnetcount(::OnB200, A; kwargs...) = DeviceColorArray(3, device_matrix(A))
selfpincount(::OnB200, A; kwargs...) = DeviceColorArray(4, device_matrix(A))

function bound_stripe(ocl::DeviceOracle, K)
    out = Vector{Float64}(undef, 2)
    check(ccall((:cpb_bound_stripe, lib), Cint, (Ptr{Cvoid}, Int64, Ptr{Float64}), ocl.h, K, out))
    return (out[1], out[2])
end

# ---- partition_stripe / pack_stripe -----------------------------------------------------------

split_code(::DynamicBottleneckSplitter) = (0, 0.0)
split_code(::DynamicTotalSplitter) = (1, 0.0)
split_code(m::BisectCostBottleneckSplitter) = (2, Float64(m.ϵ))
split_code(m::LazyBisectCostBottleneckSplitter) = (3, Float64(m.ϵ))
split_code(::ConvexTotalSplitter) = (8, 0.0)
split_code(::BisectIndexBottleneckSplitter) = (12, 0.0)
split_code(m::FlipBisectCostBottleneckSplitter) = (6, Float64(m.ϵ))          # Flip family: the secondary (decreasing) models
split_code(m::LazyFlipBisectCostBottleneckSplitter) = (7, Float64(m.ϵ))
split_code(::FlipBisectIndexBottleneckSplitter) = (13, 0.0)
split_code(::DynamicBottleneckChunker) = (10, 0.0)   # partition_stripe(A, K, ::AbstractDynamicChunker), DynamicSplitter.jl:52-87
split_code(::DynamicTotalChunker) = (11, 0.0)

split_code(::ConcaveTotalSplitter) = (9, 0.0)

function stripe_solve(dA::DeviceMatrix, K, code, ϵ, f, args...)
    ocl = DeviceOracle(dA, f, args...)
    spl = Vector{Int64}(undef, K + 1)
    GC.@preserve ocl check(ccall((:cpb_partition_stripe, lib), Cint, (Ptr{Cvoid}, Cint, Ref{CConstraint}, Float64, Int64, Ptr{Int64}),
                                 ocl.h, code, constraint(f), ϵ, K, spl))
    return SplitPartition{Int64}(K, spl)
end
function stripe_solve(dA::DeviceMatrix, K, code, ϵ, f::CountWeighted, args...)
    ocl = DeviceOracle(dA, f.f, args...)
    wcl = DeviceOracle(dA, f.w)
    spl = Vector{Int64}(undef, K + 1)
    GC.@preserve ocl wcl check(ccall((:cpb_partition_stripe_weighted, lib), Cint, (Ptr{Cvoid}, Cint, Ptr{Cvoid}, Int64, Float64, Int64, Ptr{Int64}),
                                     ocl.h, code, wcl.h, Int64(f.w_max), ϵ, K, spl))
    return SplitPartition{Int64}(K, spl)
end

# The stripe solve on a pattern that is already resident (what partition_plaid below and repeated solves use: no upload)
function partition_stripe(dA::DeviceMatrix, K, method::OnB200, args...; kwargs...)
    (code, ϵ) = split_code(method.mtd)
    return stripe_solve(dA, K, code, ϵ, method.mtd.f, args...)
end

# Many BisectIndex / Flip problems in one launch, one cluster each (cpb_partition_stripe_batch): problems is a vector of
# (A, K, OnB200(method)) or (A, K, OnB200(method), Π); each result is identical to partition_stripe(A, K, OnB200(method)[, Π]).
# Problems with the same A, model and Π objects share one oracle (a sweep over K builds it once); a host matrix is uploaded once.
function partition_stripe_batch(problems)
    mats = IdDict{Any, DeviceMatrix}()
    ocls = Dict{Tuple{UInt, UInt, UInt}, DeviceOracle}()
    hs, codes, epss, Ks, outs = Ptr{Cvoid}[], Cint[], Float64[], Int64[], Vector{Int64}[]
    for p in problems
        A, K, method = p[1], Int64(p[2]), p[3]
        Π = length(p) >= 4 ? p[4] : nothing
        (code, ϵ) = split_code(method.mtd)
        code in (12, 6, 7, 13) || throw(ArgumentError("partition_stripe_batch takes the BisectIndex and Flip splitters only"))
        dA = get!(() -> device_matrix(A), mats, A)
        ocl = get!(() -> DeviceOracle(dA, method.mtd.f, Π), ocls, (objectid(A), objectid(method.mtd.f), objectid(Π)))
        push!(hs, ocl.h); push!(codes, code); push!(epss, ϵ); push!(Ks, K); push!(outs, Vector{Int64}(undef, K + 1))
    end
    ptrs = [pointer(o) for o in outs]
    GC.@preserve mats ocls outs check(ccall((:cpb_partition_stripe_batch, lib), Cint,
                                            (Int64, Ptr{Ptr{Cvoid}}, Ptr{Cint}, Ptr{Float64}, Ptr{Int64}, Ptr{Ptr{Int64}}),
                                            length(hs), hs, codes, epss, Ks, ptrs))
    return [SplitPartition{Int64}(K, o) for (K, o) in zip(Ks, outs)]
end

# partition_plaid(A, K, AlternatingPartitioner(OnB200(m1), OnB200(m2), ...)) (src/AlternatingPartitioner.jl:18-32): A is
# uploaded ONCE, adjointpattern runs on the device, every stripe solve takes the resident handles -- the reference's
# `adj_A = adjointpattern(A)` reuse seam, kept on the device.  A caller-supplied adj_A (host or device) is honoured.
function partition_plaid(A::Union{SparseMatrixCSC, DeviceMatrix}, K, method::AlternatingPartitioner{<:Tuple{Vararg{OnB200}}}; adj_A = nothing, kwargs...)
    dA = device_matrix(A)
    dT = adj_A === nothing ? adjointpattern(dA) : device_matrix(adj_A)
    Φ = partition_stripe(dA, K, method.mtds[1])
    Π = partition_stripe(dT, K, method.mtds[2], Φ)
    for (i, mtd) in enumerate(method.mtds[3:end])
        if isodd(i)
            Φ = partition_stripe(dA, K, mtd, Π)
        else
            Π = partition_stripe(dT, K, mtd, Φ)
        end
    end
    return (Π, Φ)
end
function partition_plaid(A::Union{SparseMatrixCSC, DeviceMatrix}, K, method::SymmetricPartitioner{<:Tuple{Vararg{OnB200}}}; adj_A = nothing, kwargs...)
    dA = device_matrix(A)
    Π = partition_stripe(dA, K, method.mtds[1])
    if length(method.mtds) > 1
        dT = adj_A === nothing ? adjointpattern(dA) : device_matrix(adj_A)
        for (i, mtd) in enumerate(method.mtds[2:end])
            Π = partition_stripe(isodd(i) ? dA : dT, K, mtd, Π)
        end
    end
    return (Π, Π)
end

# ---- one solve over several GPUs (one Julia process per GPU; cpb_comm_*, cpb_partition_stripe_sharded) ------------
# rank 0: id = comm_unique_id(); ship the 128 bytes to the other ranks (MPI.bcast, a file, ...); every rank: comm_init
function comm_unique_id()
    id = Vector{UInt8}(undef, 128)
    check(ccall((:cpb_comm_unique_id, lib), Cint, (Ptr{UInt8},), id))
    return id
end
init(device::Integer) = check(ccall((:cpb_init, lib), Cint, (Cint,), device))
comm_init(id::Vector{UInt8}, rank::Integer, world::Integer) = check(ccall((:cpb_comm_init, lib), Cint, (Ptr{UInt8}, Cint, Cint), id, rank, world))
comm_destroy() = check(ccall((:cpb_comm_destroy, lib), Cint, ()))
# A pattern spread over the ranks (cpb_sharded): the column offsets on every rank, each rank's block of rowval.  Collective:
# every rank calls it with the same A; each uploads only its block of rowval.  Free it with close_sharded on every rank.
mutable struct ShardedMatrix
    h::Ptr{Cvoid}
    m::Int64
    n::Int64
end
function ShardedMatrix(A::SparseMatrixCSC{Tv, Int64}) where {Tv}
    (m, n) = size(A)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    GC.@preserve A check(ccall((:cpb_sharded_matrix_create, lib), Cint, (Int64, Int64, Int64, Ptr{Int64}, Ptr{Int64}, Cint, Ref{Ptr{Cvoid}}),
                               m, n, nnz(A), A.colptr, A.rowval, 0, h))
    return ShardedMatrix(h[], m, n)
end
function close_sharded(S::ShardedMatrix)
    S.h == C_NULL || ccall((:cpb_sharded_matrix_destroy, lib), Cvoid, (Ptr{Cvoid},), S.h)
    S.h = C_NULL
end
# adjointpattern of the sharded pattern (collective): the transpose with the same blocks of CSC positions
function adjointpattern(S::ShardedMatrix)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:cpb_sharded_adjointpattern, lib), Cint, (Ptr{Cvoid}, Ref{Ptr{Cvoid}}), S.h, h))
    return ShardedMatrix(h[], S.n, S.m)
end
# (colptr, this rank's block of rowval, q_lo, q_hi): 1-based indices, 0-based half-open block of CSC positions
function host_block(S::ShardedMatrix)
    lo, hi = Ref{Int64}(0), Ref{Int64}(0)
    check(ccall((:cpb_sharded_matrix_get, lib), Cint, (Ptr{Cvoid}, Ptr{Int64}, Ptr{Int64}, Ref{Int64}, Ref{Int64}), S.h, C_NULL, C_NULL, lo, hi))
    colptr, rowval = Vector{Int64}(undef, S.n + 1), Vector{Int64}(undef, hi[] - lo[])
    check(ccall((:cpb_sharded_matrix_get, lib), Cint, (Ptr{Cvoid}, Ptr{Int64}, Ptr{Int64}, Ptr{Int64}, Ptr{Int64}), S.h, colptr,
                isempty(rowval) ? C_NULL : pointer(rowval), C_NULL, C_NULL))
    return (colptr, rowval, lo[], hi[])
end
const ShardedSplitter = OnB200{<:Union{BisectCostBottleneckSplitter, LazyBisectCostBottleneckSplitter}}
# collective: ONE stripe solve over all ranks, AffineConnectivityModel or AffineMonotonizedSymmetricConnectivityModel (square
# A); the library refuses any other model on every rank alike
function partition_stripe_sharded(S::ShardedMatrix, K, method::ShardedSplitter, args...)
    (code, ϵ) = split_code(method.mtd)
    (cm, keep) = cmodel(method.mtd.f, 0, 0)
    spl = Vector{Int64}(undef, K + 1)
    GC.@preserve keep check(ccall((:cpb_partition_stripe_sharded, lib), Cint, (Ptr{Cvoid}, Ref{CModel}, Cint, Float64, Int64, Ptr{Int64}), S.h, cm, code, ϵ, K, spl))
    return SplitPartition{Int64}(K, spl)
end
function partition_stripe_sharded(A::SparseMatrixCSC{Tv, Int64}, K, method::ShardedSplitter) where {Tv}
    S = ShardedMatrix(A)
    try
        return partition_stripe_sharded(S, K, method)
    finally
        close_sharded(S)
    end
end
# partition_plaid(A, K, AlternatingPartitioner(...)) (src/AlternatingPartitioner.jl:18-32) with every stripe solve sharded
# over the ranks; the transpose is built once (cpb_sharded_adjointpattern) unless adj_A is given.  Collective.
function partition_plaid_sharded(A::Union{SparseMatrixCSC, ShardedMatrix}, K, method::AlternatingPartitioner{<:Tuple{Vararg{ShardedSplitter}}}; adj_A = nothing)
    S = A isa ShardedMatrix ? A : ShardedMatrix(A)
    T = adj_A === nothing ? adjointpattern(S) : (adj_A isa ShardedMatrix ? adj_A : ShardedMatrix(adj_A))
    try
        Φ = partition_stripe_sharded(S, K, method.mtds[1])
        Π = partition_stripe_sharded(T, K, method.mtds[2])
        for (i, mtd) in enumerate(method.mtds[3:end])
            if isodd(i)
                Φ = partition_stripe_sharded(S, K, mtd)
            else
                Π = partition_stripe_sharded(T, K, mtd)
            end
        end
        return (Π, Φ)
    finally
        T === adj_A || close_sharded(T)
        S === A || close_sharded(S)
    end
end

function partition_stripe(A::SparseMatrixCSC{Tv, Int64}, K, method::OnB200, args...; kwargs...) where {Tv}
    dA = DeviceMatrix(A)
    (code, ϵ) = split_code(method.mtd)
    return stripe_solve(dA, K, code, ϵ, method.mtd.f, args...)
end

pack_code(m::DynamicTotalChunker) = (0, m.f, 0.0, 0)
pack_code(m::ConvexTotalChunker) = (1, m.f, 0.0, 0)
pack_code(m::ConcaveTotalChunker) = (2, m.f, 0.0, 0)
pack_code(m::OverlapChunker) = (3, nothing, m.ρ, m.w_max)
pack_code(m::StrictChunker) = (4, nothing, 0.0, m.w_max)
pack_code(m::EquiChunker) = (5, nothing, 0.0, m.w)

function pack_stripe(A::SparseMatrixCSC{Tv, Int64}, method::OnB200, args...; n_nets = nothing, kwargs...) where {Tv}
    (m, n) = size(A)
    dA = DeviceMatrix(A)
    (code, f, ρ, w_max) = pack_code(method.mtd)
    con = constraint(f)
    ocl = f === nothing ? nothing : DeviceOracle(dA, f, args...; w_tab = con.enabled == 1 ? min(n, con.w_max ÷ max(con.w_coef[2], 1) + 1) : n)
    spl = Vector{Int64}(undef, n + 1)
    nn = Vector{Int64}(undef, max(n, 1))
    K = Ref{Int64}(0)
    check(ccall((:cpb_pack_stripe, lib), Cint,
                (Ptr{Cvoid}, Ptr{Cvoid}, Cint, Ref{CConstraint}, Float64, Int64, Ptr{Int64}, Ref{Int64}, Ptr{Int64}),
                dA.h, ocl === nothing ? C_NULL : ocl.h, code, con, ρ, w_max, spl, K, nn))
    if n_nets isa Ref
        n_nets[] = nn[1:K[]]
    end
    return SplitPartition{Int64}(K[], resize!(spl, K[] + 1))
end

# ---- SparsePrefixMatrices.jl on the device: dominancecount / dominancesum / rookcount! / rooksum! --------------------
# (src/SparsePrefixMatrices.jl:31-58, 440-460, 840-851, 1056-1063).  One handle type; `C[i, j]` as in the reference.
# The device takes the place of the hint argument: `dominancecount(OnB200(nothing), A)`.
mutable struct DevicePrefixMatrix{Tv} <: AbstractMatrix{Tv}
    h::Ptr{Cvoid}
    m::Int
    n::Int
    summed::Bool
    function DevicePrefixMatrix{Tv}(m, n, N, pos, idx::Vector{Int64}, val) where {Tv}
        h = Ref{Ptr{Cvoid}}(C_NULL)
        GC.@preserve pos idx val check(ccall((:cpb_prefix_create, lib), Cint,
            (Int64, Int64, Int64, Ptr{Int64}, Ptr{Int64}, Ptr{Int64}, Ref{Ptr{Cvoid}}), m, n, N,
            pos === nothing ? C_NULL : pointer(pos), idx, val === nothing ? C_NULL : Ptr{Int64}(pointer(val)), h))
        finalizer(x -> ccall((:cpb_prefix_destroy, lib), Cvoid, (Ptr{Cvoid},), x.h), new{Tv}(h[], m, n, val !== nothing))
    end
end
Base.size(P::DevicePrefixMatrix) = (P.m + 1, P.n + 1)
function Base.getindex(P::DevicePrefixMatrix{Tv}, i::Integer, j::Integer) where {Tv}
    out = Ref{Int64}(0)
    check(ccall((:cpb_prefix_query, lib), Cint, (Ptr{Cvoid}, Int64, Ref{Int64}, Ref{Int64}, Ptr{Int64}, Ptr{Int64}),
                P.h, 1, Int64(i), Int64(j), P.summed ? C_NULL : out, P.summed ? out : C_NULL))
    return reinterpret(Tv, out[])
end
dominancecount(::OnB200, A::SparseMatrixCSC{Tv, Int64}; kwargs...) where {Tv} =
    DevicePrefixMatrix{Int64}(size(A)..., nnz(A), A.colptr, A.rowval, nothing)
dominancesum(::OnB200, A::SparseMatrixCSC{Tv, Int64}; kwargs...) where {Tv <: Union{Int64, UInt64}} =
    DevicePrefixMatrix{Tv}(size(A)..., nnz(A), A.colptr, A.rowval, A.nzval)
rookcount!(::OnB200, N, idx::Vector{Int64}; kwargs...) = DevicePrefixMatrix{Int64}(N, N, N, nothing, idx, nothing)
rooksum!(::OnB200, N, idx::Vector{Int64}, val::Vector{Tv}; kwargs...) where {Tv <: Union{Int64, UInt64}} =
    DevicePrefixMatrix{Tv}(N, N, N, nothing, idx, val)

# pack_plaid needs no glue: AlternatingPacker(OnB200(mtd1), OnB200(mtd2)) alternates pack_stripe calls on A and
# adjointpattern(A) (src/AlternatingPacker.jl:6-53); partition_plaid has the resident-handle methods above.

end # module
