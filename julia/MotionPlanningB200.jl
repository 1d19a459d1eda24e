# MotionPlanningB200.jl -- the binding a MotionPlanning.jl maintainer would add to switch the hot
# path to libmpb200.so (include/mpb200.h).  Julia-0.5-era syntax to match the reference; it cannot
# be executed in this repository's containers (no julia): it is complete, loadable-as-written code (no
# stubs), every ccall signature and struct layout below is checked against the header by tests/test_abi.py,
# and the same ABI is exercised from plain C by tests/c_abi_driver.c.
#
# Seams used (all already present in the reference):
#   * helper_data_structures(V, dist) is overloaded per metric (geometric.jl:14, linearquadratic.jl:68)
#   * ImmutableNNC{T}(D::SparseMatrixCSC{T,Int}, r) is served by viewcol (nearneighbors.jl:23-28,128)
#   * SweptCollisionChecker subtypes implement is_free_state / is_free_motion and carry `count`
#     (collisioncheckers.jl:4-6, robots2D.jl:5-14, boxesND.jl:15-27)
module MotionPlanningB200

using MotionPlanning
import MotionPlanning: is_free_state, is_free_motion, is_free_path, helper_data_structures, inball!, inballF!, inballB!
using StaticArrays

const LIB = "libmpb200"
check(rc) = rc == 0 || error(unsafe_string(ccall((:mpb200_last_error, LIB), Cstring, ())))
init(device = 0) = check(ccall((:mpb200_init, LIB), Cint, (Cint,), device))

# ---- sample sets -------------------------------------------------------------------------------
type B200Samples
    h::Ptr{Void}
end
function B200Samples{S<:SVector}(V::Vector{S})
    h = Ref{Ptr{Void}}(C_NULL)
    M = statevec2mat(V)                      # zero-copy d x N view (primitivetypes.jl:21-23)
    check(ccall((:mpb200_samples_create, LIB), Cint, (Ptr{Float64}, Int64, Cint, Ref{Ptr{Void}}),
                M, size(M, 2), size(M, 1), h))
    s = B200Samples(h[])
    finalizer(s, x -> ccall((:mpb200_samples_destroy, LIB), Cint, (Ptr{Void},), x.h))
    s
end

# ---- Euclidean: the whole ImmutableNNC table in one call ------------------------------------------
"Precompute every r-ball on the GPU and install it as the sample set's ImmutableNNC (nearneighbors.jl:128)."
function precompute_inball!(NN::MetricNN, r::Float64)
    s = B200Samples(NN.V)
    t = Ref{Ptr{Void}}(C_NULL); nnz = Ref{Int64}(0)
    check(ccall((:mpb200_inball_build, LIB), Cint, (Ptr{Void}, Float64, Ref{Ptr{Void}}, Ref{Int64}), s.h, r, t, nnz))
    N = length(NN.V)
    colptr = Array(Int64, N + 1); rowval = Array(Int64, nnz[]); nzval = Array(Float64, nnz[])
    check(ccall((:mpb200_table_fetch, LIB), Cint, (Ptr{Void}, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}),
                t[], colptr, rowval, nzval))
    D = SparseMatrixCSC(N, N, colptr, rowval, nzval)   # fields cross unchanged: 1-based Int64 / Float64
    NNi = MetricNN(NN.V, NN.dist, NN.init, ImmutableNNC(D, fill(r, N)), NN.DS, NN.US)
    NNi, s, t[]
end

# ---- state spaces: BoundedStateSpace bounds + State2Workspace -> mpb200_space_desc ---------------------
# C layout of mpb200_space_desc (include/mpb200.h): int32 n; double* lo; double* hi; int32 s2w_kind; int32 dw;
# int32* inds; double* C.  The struct holds POINTERS into Julia arrays, so those arrays travel with it
# (`keep`) and the struct is handed to ccall by reference.
immutable SpaceDescC
    n::Int32
    lo::Ptr{Float64}
    hi::Ptr{Float64}
    s2w_kind::Int32
    dw::Int32
    inds::Ptr{Int32}
    C::Ptr{Float64}
end
type SpaceDesc
    c::Base.RefValue{SpaceDescC}
    keep::Vector{Any}                       # lo, hi, inds, C: rooted for as long as the descriptor lives
end
s2w_fields(::Identity, n) = (Int32(0), Int32(n), Int32[], Float64[])
s2w_fields(w::VectorView, n) = (Int32(1), Int32(length(w.inds)), Int32[i - 1 for i in w.inds], Float64[])   # 0-based
s2w_fields(w::OutputMatrix, n) = (Int32(2), Int32(size(w.C, 1)), Int32[], Float64[w.C[i, j] for i in 1:size(w.C, 1), j in 1:size(w.C, 2)][:])  # column-major
"statespaces.jl:29-34 (bounds) and :45-60 (State2Workspace) as the C descriptor"
function space_desc(SS::BoundedStateSpace)
    lo = Float64[SS.lo...]; hi = Float64[SS.hi...]
    kind, dw, inds, C = s2w_fields(SS.s2w, length(lo))
    d = SpaceDescC(Int32(length(lo)), pointer(lo), pointer(hi), kind, dw,
                   isempty(inds) ? Ptr{Int32}(C_NULL) : pointer(inds), isempty(C) ? Ptr{Float64}(C_NULL) : pointer(C))
    SpaceDesc(Ref(d), Any[lo, hi, inds, C])
end
# a checker used without a state space (robots2D.jl:12-13 call forms): no bounds, identity map
space_desc(n::Int) = (lo = fill(-Inf, n); hi = fill(Inf, n);
                      SpaceDesc(Ref(SpaceDescC(Int32(n), pointer(lo), pointer(hi), Int32(0), Int32(n), C_NULL, C_NULL)), Any[lo, hi]))

# ---- collision checkers ----------------------------------------------------------------------------
# C layout of mpb200_obstacles2d_desc
immutable Obstacles2DDescC
    n_gates::Int32
    gate_parent::Ptr{Int32}
    gate_aabb::Ptr{Float64}
    n_shapes::Int32
    shape_kind::Ptr{Int32}
    shape_gate::Ptr{Int32}
    shape_off::Ptr{Int32}
    data::Ptr{Float64}
    flags::Int32
end

"""
Flatten a shape tree into the arrays of mpb200_obstacles2d_desc.  Compound2D nodes (SAT2D.jl:82-96) become AABB
gates, parent before child; Circle (:12-25) -> [c; r; xrange; yrange]; Polygon (:29-51) -> [xrange; yrange; points;
normals; nextrema] -- everything already PRECOMPUTED by the reference's own constructors, so the device evaluates the
predicates on exactly the numbers Julia would (normalize()'s rounding included).
"""
function pack(shape::Shape2D)
    gate_parent = Int32[]; gate_aabb = Float64[]
    kinds = Int32[]; gates = Int32[]; offs = Int32[0]; data = Float64[]
    function walk(s::Compound2D, parent)
        g = Int32(length(gate_parent))
        push!(gate_parent, Int32(parent))
        append!(gate_aabb, [s.xrange[1], s.xrange[2], s.yrange[1], s.yrange[2]])
        for p in s.parts
            walk(p, g)
        end
    end
    function walk(s::Circle, parent)
        push!(kinds, Int32(0)); push!(gates, Int32(parent))
        append!(data, [s.c[1], s.c[2], s.r, s.xrange[1], s.xrange[2], s.yrange[1], s.yrange[2]])
        push!(offs, Int32(length(data)))
    end
    function walk(s::Polygon, parent)
        push!(kinds, Int32(1)); push!(gates, Int32(parent))
        append!(data, [s.xrange[1], s.xrange[2], s.yrange[1], s.yrange[2]])
        for p in s.points;   append!(data, [p[1], p[2]]); end
        for n in s.normals;  append!(data, [n[1], n[2]]); end
        for e in s.nextrema; append!(data, [e[1], e[2]]); end
        push!(offs, Int32(length(data)))
    end
    walk(s::Shape2D, parent) = error("obstacles must be Circle, Polygon or Compound2D")   # e.g. Line
    walk(shape, -1)
    gate_parent, gate_aabb, kinds, gates, offs, data
end

type B200PointRobot2D{S<:Shape2D} <: SweptCollisionChecker
    obstacles::S                 # host-side shapes (constructors, inflate, closest, plotting stay in Julia)
    h::Ptr{Void}
    count::Int
end
"PointRobot2D(obstacles) (robots2D.jl:5-10) with the obstacle table resident on the GPU"
function B200PointRobot2D(obstacles::Shape2D; fixed_point_test = false)
    gp, ga, kinds, gates, offs, data = pack(obstacles)
    d = Ref(Obstacles2DDescC(Int32(length(gp)), pointer(gp), pointer(ga), Int32(length(kinds)), pointer(kinds),
                             pointer(gates), pointer(offs), pointer(data), Int32(fixed_point_test ? 1 : 0)))
    h = Ref{Ptr{Void}}(C_NULL)
    check(ccall((:mpb200_obstacles2d_create, LIB), Cint, (Ref{Obstacles2DDescC}, Ref{Ptr{Void}}), d, h))   # copies the arrays
    CC = B200PointRobot2D(obstacles, h[], 0)
    finalizer(CC, x -> ccall((:mpb200_obstacles_destroy, LIB), Cint, (Ptr{Void},), x.h))
    CC
end

type B200PointRobotNDBoxes{N,T} <: SweptCollisionChecker
    boxes::Vector{BoxBounds{N,T}}
    h::Ptr{Void}
    count::Int
end
"PointRobotNDBoxes(boxes) (boxesND.jl:15-21); lo / hi cross box-major M x d"
function B200PointRobotNDBoxes{N,T}(boxes::Vector{BoxBounds{N,T}})
    M = length(boxes)
    lo = Float64[boxes[k].lo[i] for i in 1:N, k in 1:M][:]     # box k occupies lo[(k-1)N+1 : kN]
    hi = Float64[boxes[k].hi[i] for i in 1:N, k in 1:M][:]
    h = Ref{Ptr{Void}}(C_NULL)
    check(ccall((:mpb200_boxes_create, LIB), Cint, (Ptr{Float64}, Ptr{Float64}, Cint, Cint, Ref{Ptr{Void}}), lo, hi, M, N, h))
    CC = B200PointRobotNDBoxes(boxes, h[], 0)
    finalizer(CC, x -> ccall((:mpb200_obstacles_destroy, LIB), Cint, (Ptr{Void},), x.h))
    CC
end
typealias B200Checker Union{B200PointRobot2D, B200PointRobotNDBoxes}

# the host-side conveniences keep working through the wrapped reference objects (robots2D.jl:21-26, boxesND.jl:30-34)
MotionPlanning.inflate(CC::B200PointRobot2D, eps; roundcorners = true) =
    eps > 0 ? B200PointRobot2D(inflate(CC.obstacles, eps, roundcorners = roundcorners)) : CC
MotionPlanning.addobstacle(CC::B200PointRobot2D, o::Shape2D) = B200PointRobot2D(Compound2D(CC.obstacles, o))
MotionPlanning.addblocker(CC::B200PointRobot2D, p::AbstractVector, r) = addobstacle(CC, Circle(p, r))
MotionPlanning.inflate{N,T}(CC::B200PointRobotNDBoxes{N,T}, eps) =
    eps > 0 ? B200PointRobotNDBoxes([inflate(B, T(eps)) for B in CC.boxes]) : CC
MotionPlanning.addobstacle(CC::B200PointRobotNDBoxes, o) = B200PointRobotNDBoxes(vcat(CC.boxes, BoxBounds(o)))
MotionPlanning.addblocker(CC::B200PointRobotNDBoxes, v::AbstractVector, r) = addobstacle(CC, BoxBounds(v - r, v + r))

# state-level calls (fmt.jl:24,34,75 pass states): batches of one.  With a state space the wrappers of
# statespaces.jl:151-158 (bounds, state2workspace, waypoints) run on the device as well.
function states_free(V::Matrix{Float64}, CC::B200Checker, sd::SpaceDesc)
    out = Array(UInt8, size(V, 2))
    check(ccall((:mpb200_states_free, LIB), Cint, (Ptr{Float64}, Int64, Cint, Ptr{Void}, Ref{SpaceDescC}, Ptr{UInt8}),
                V, size(V, 2), size(V, 1), CC.h, sd.c, out))
    out
end
function segments_free(V::Matrix{Float64}, W::Matrix{Float64}, CC::B200Checker, sd::SpaceDesc)
    out = Array(UInt8, size(V, 2))
    check(ccall((:mpb200_segments_free, LIB), Cint,
                (Ptr{Float64}, Ptr{Float64}, Int64, Cint, Ptr{Void}, Ref{SpaceDescC}, Ptr{UInt8}),
                V, W, size(V, 2), size(V, 1), CC.h, sd.c, out))
    out
end
col(v::AbstractVector) = reshape(Float64[v...], length(v), 1)
is_free_state(v::AbstractVector, CC::B200Checker, SS::StateSpace) = states_free(col(v), CC, space_desc(SS))[1] != 0
is_free_state(v::AbstractVector, CC::B200Checker) = states_free(col(v), CC, space_desc(length(v)))[1] != 0
function is_free_motion(v::AbstractVector, w::AbstractVector, CC::B200Checker, SS::StateSpace)
    # Euclidean spaces: collision_waypoints = (v, w) (geometric.jl:20).  LinearQuadratic spaces go through
    # mpb200_lq_motions_free (5 waypoints of the optimal trajectory, linearquadratic.jl:85-88) -- see below.
    in_state_space(v, SS) && (CC.count += 1)         # the wrapper short-circuits before the segment test (statespaces.jl:155-157)
    segments_free(col(v), col(w), CC, space_desc(SS))[1] != 0
end
is_free_motion(v::AbstractVector, w::AbstractVector, CC::B200Checker) =
    (CC.count += 1; segments_free(col(v), col(w), CC, space_desc(length(v)))[1] != 0)
"robots2D.jl:15-20 / statespaces.jl:159-160: every consecutive pair, as ONE batch (the result is the same conjunction)"
function is_free_path(path::Path, CC::B200Checker)
    length(path) < 2 && return true
    V = hcat([Float64[p...] for p in path[1:end-1]]...); W = hcat([Float64[p...] for p in path[2:end]]...)
    CC.count += size(V, 2)
    all(segments_free(V, W, CC, space_desc(size(V, 1))) .!= 0)
end
function is_free_path(path::Path, CC::B200Checker, SS::StateSpace)
    length(path) < 2 && return true
    V = hcat([Float64[p...] for p in path[1:end-1]]...); W = hcat([Float64[p...] for p in path[2:end]]...)
    CC.count += count(i -> in_state_space(path[i], SS), 1:length(path)-1)
    all(segments_free(V, W, CC, space_desc(SS)) .!= 0)
end
# LinearQuadratic spaces: the motion V[y] -> V[x] is checked along the optimal trajectory
function is_free_motion{S,M<:LinearQuadratic}(v::AbstractVector, w::AbstractVector, CC::B200Checker,
                                              SS::BoundedStateSpace{S,M}, lq::Ptr{Void})
    out = Ref{UInt8}(0); checks = Ref{Int64}(0)
    sd = space_desc(SS)
    check(ccall((:mpb200_lq_motions_free, LIB), Cint,
                (Ptr{Void}, Float64, Ptr{Float64}, Ptr{Float64}, Int64, Ptr{Void}, Ref{SpaceDescC}, Ref{UInt8}, Ref{Int64}),
                lq, SS.dist.cmax, col(v), col(w), 1, CC.h, sd.c, out, checks))
    CC.count += checks[]
    out[] != 0
end

# ---- the drop-in change in fmtstar! ------------------------------------------------------------------
# Batched tables: F (point validity) and E (edge validity, aligned with the backward table: stored
# entry k of column x, row y  <=>  is_free_motion(V[y], V[x], CC, SS)).
#   sd = space_desc(SS)
#   F = BitVector(N); check(ccall((:mpb200_points_free, LIB), Cint, (Ptr{Void},Ptr{Void},Ref{SpaceDescC},Ptr{UInt64}),
#                                 s.h, CC.h, sd.c, F.chunks))
#   E = BitVector(nnz); checks = Ref{Int64}(0)
#   check(ccall((:mpb200_edges_free, LIB), Cint, (Ptr{Void},Ptr{Void},Ptr{Void},Ref{SpaceDescC},Ptr{UInt64},Ref{Int64}),
#               s.h, t, CC.h, sd.c, E.chunks, checks))
# and fmt.jl:72-75 becomes (one changed line; y_idx is already computed there):
#   neighborhood = nearB(P.V, x, r, H)          # still a viewcol of the ImmutableNNC
#   c_min, y_idx = findmin(C[nonzeroinds(neighborhood)] + nonzeros(neighborhood))
#   k = P.V.cache.D.colptr[x] - 1 + findnth(H[rowvals_of_column_x], y_idx)   # position of y_min in column x
#   if E[k]                                       # was: is_free_motion(P.V[y_min], P.V[x], P.CC, P.SS)

# ---- sample_free! on the device (sampling.jl:23-37) -------------------------------------------------------
# The uniform bulk of the sample set is drawn, filtered with is_free_state and compacted on the GPU; the handle
# is kept for the table builds, the host copy feeds P.V.  (Own Philox stream: deterministic in `seed`, not
# Julia's global RNG.)
function sample_free_b200(SS::StateSpace, CC::B200Checker, N::Int, seed::UInt64)
    d = dim(SS)
    M = Array(Float64, d, N)
    h = Ref{Ptr{Void}}(C_NULL); used = Ref{Int64}(0)
    sd = space_desc(SS)
    check(ccall((:mpb200_sample_free, LIB), Cint,
                (Ptr{Void}, Ref{SpaceDescC}, Int64, UInt64, Int32, Ref{Ptr{Void}}, Ptr{Float64}, Ref{Int64}),
                CC.h, sd.c, N, seed, Int32(1), h, M, used))   # 1 = Morton numbering
    s = B200Samples(h[])                              # adopt the handle
    finalizer(s, x -> ccall((:mpb200_samples_destroy, LIB), Cint, (Ptr{Void},), x.h))
    reinterpret(SVector{d,Float64}, M, (N,)), s, used[]
end

# ---- linear-quadratic (ControlNN) ---------------------------------------------------------------------
function helper_data_structures{S}(V::Vector{S}, M::LinearQuadratic, backend::Type{Val{:b200}})
    s = B200Samples(V)
    lq = Ref{Ptr{Void}}(C_NULL)
    b = M.bvp
    check(ccall((:mpb200_lq_create, LIB), Cint,
                (Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Cint, Cint, Ref{Ptr{Void}}),
                b.A, b.B, b.c, b.R, size(b.A, 1), size(b.B, 2), lq))
    tF = Ref{Ptr{Void}}(C_NULL); tB = Ref{Ptr{Void}}(C_NULL); nF = Ref{Int64}(0); nB = Ref{Int64}(0)
    check(ccall((:mpb200_lq_inball_build, LIB), Cint,
                (Ptr{Void}, Ptr{Void}, Float64, Ref{Ptr{Void}}, Ref{Ptr{Void}}, Ref{Int64}, Ref{Int64}),
                s.h, lq[], M.cmax, tF, tB, nF, nB))
    fetch(t, nnz) = begin
        N = length(V)
        cp = Array(Int64, N + 1); rv = Array(Int64, nnz); nz = Array(Float64, nnz)
        check(ccall((:mpb200_table_fetch, LIB), Cint, (Ptr{Void}, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}), t, cp, rv, nz))
        SparseMatrixCSC(N, N, cp, rv, nz)
    end
    US = EmptyControlCache()
    BruteDistanceDS(fetch(tF[], nF[])), US, BruteDistanceDS(fetch(tB[], nB[])), US   # DSF, USF, DSB, USB (:73-76)
end

# ---- chopped-metric car spaces (simplecars.jl) ------------------------------------------------------------
# helper_data_structures(V, ::ChoppedMetric{ReedsSheppExact}) / (V, ::ChoppedQuasiMetric{DubinsExact}) build a KD-tree
# over (x, y) and every inball evaluates the exact metric on its candidates (simplecars.jl:42-52,
# nearneighbors.jl:185-198); here the whole forward (and, for Dubins, backward) table is built at once and served as
# ImmutableNNC caches.  kind: 0 = Reeds-Shepp, 1 = Dubins (MPB200_CAR_*).
car_kind(::ReedsSheppExact) = Int32(0)
car_kind(::DubinsExact) = Int32(1)
function fetch_table(t::Ptr{Void}, N::Int, nnz::Int64)
    cp = Array(Int64, N + 1); rv = Array(Int64, nnz); nz = Array(Float64, nnz)
    check(ccall((:mpb200_table_fetch, LIB), Cint, (Ptr{Void}, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}), t, cp, rv, nz))
    SparseMatrixCSC(N, N, cp, rv, nz)
end
function precompute_inball!{R<:ReedsSheppExact}(NN::MetricNN, M::ChoppedMetric{R}, r::Float64)
    s = B200Samples(NN.V)                                   # SE2State is a FieldVector: 3 x N Float64
    tF = Ref{Ptr{Void}}(C_NULL); nF = Ref{Int64}(0)
    check(ccall((:mpb200_car_inball_build, LIB), Cint,
                (Ptr{Void}, Int32, Float64, Float64, Float64, Ref{Ptr{Void}}, Ptr{Void}, Ref{Int64}, Ptr{Void}),
                s.h, car_kind(M.m), M.m.r, r, M.chopval, tF, C_NULL, nF, C_NULL))
    N = length(NN.V)
    MetricNN(NN.V, NN.dist, NN.init, ImmutableNNC(fetch_table(tF[], N, nF[]), fill(r, N)), NN.DS, NN.US), s, tF[]
end
function precompute_inball!{D<:DubinsExact}(NN::QuasiMetricNN, M::ChoppedQuasiMetric{D}, r::Float64)
    s = B200Samples(NN.V)
    tF = Ref{Ptr{Void}}(C_NULL); tB = Ref{Ptr{Void}}(C_NULL); nF = Ref{Int64}(0); nB = Ref{Int64}(0)
    check(ccall((:mpb200_car_inball_build, LIB), Cint,
                (Ptr{Void}, Int32, Float64, Float64, Float64, Ref{Ptr{Void}}, Ref{Ptr{Void}}, Ref{Int64}, Ref{Int64}),
                s.h, car_kind(M.m), M.m.r, r, M.chopval, tF, tB, nF, nB))
    N = length(NN.V)
    QuasiMetricNN(NN.V, NN.dist, NN.init, ImmutableNNC(fetch_table(tF[], N, nF[]), fill(r, N)),
                  ImmutableNNC(fetch_table(tB[], N, nB[]), fill(r, N)), NN.DSF, NN.USF, NN.DSB, NN.USB), s, tF[], tB[]
end
# is_free_motion(v, w, CC, SS) over the arc waypoints (statespaces.jl:153-158, simplecars.jl:71-82)
function is_free_motion{S,M<:ChoppedPreMetric}(v::SE2State, w::SE2State, CC::B200Checker, SS::BoundedStateSpace{S,M})
    sd = space_desc(SS); out = Array(UInt8, 1); checks = Ref{Int64}(0); m = SS.dist.m
    check(ccall((:mpb200_car_motions_free, LIB), Cint,
                (Int32, Float64, Float64, Ptr{Float64}, Ptr{Float64}, Int64, Ptr{Void}, Ref{SpaceDescC}, Ptr{UInt8}, Ref{Int64}),
                car_kind(m), m.r, m.s, Float64[v...], Float64[w...], 1, CC.h, sd.c, out, checks))
    CC.count += checks[]
    out[1] != 0
end
# steering_control(d, v, w) (simplecars.jl:69-70) as the reference's ZeroOrderHoldControl
function steering_control_b200(m::SimpleCarMetric, v::SE2State, w::SE2State)
    cost = Array(Float64, 1); nseg = Array(Int32, 1); segs = Array(Float64, 3, 5)
    check(ccall((:mpb200_car_steer, LIB), Cint,
                (Int32, Float64, Float64, Ptr{Float64}, Ptr{Float64}, Int64, Ptr{Float64}, Ptr{Int32}, Ptr{Float64}),
                car_kind(m), m.r, m.s, Float64[v...], Float64[w...], 1, cost, nseg, segs))
    cost[1], [StepControl(segs[1, i], SVector(segs[2, i], segs[3, i])) for i in 1:nseg[1]]
end
# validity of every stored edge (row y -> column x  <=>  is_free_motion(V[y], V[x], CC, SS)) as a BitVector
function car_edges_free(s::B200Samples, t::Ptr{Void}, nnz::Int64, CC::B200Checker, SS::BoundedStateSpace)
    sd = space_desc(SS); bits = BitVector(nnz); checks = Ref{Int64}(0); m = SS.dist.m
    check(ccall((:mpb200_car_edges_free, LIB), Cint,
                (Ptr{Void}, Ptr{Void}, Int32, Float64, Float64, Ptr{Void}, Ref{SpaceDescC}, Ptr{UInt64}, Ref{Int64}),
                s.h, t, car_kind(m), m.r, m.s, CC.h, sd.c, bits.chunks, checks))
    bits, checks[]
end

# ---- k-nearest connections (names exported at nearneighbors.jl:9-11, used at fmt.jl:17-19, defined nowhere) ------
# table operations on any neighbour table: the k best entries of every column, and the mutual neighbourhoods
# knnF(v) U { w : v in knnB(w) }; `short` = columns of t that held fewer than k entries (grow r and rebuild until 0)
function table_knn(t::Ptr{Void}, k::Int)
    out = Ref{Ptr{Void}}(C_NULL); nnz = Ref{Int64}(0); short = Ref{Int64}(0)
    check(ccall((:mpb200_table_knn, LIB), Cint, (Ptr{Void}, Cint, Ref{Ptr{Void}}, Ref{Int64}, Ref{Int64}), t, k, out, nnz, short))
    out[], nnz[], short[]
end
function table_union_transpose(a::Ptr{Void}, b::Ptr{Void})
    out = Ref{Ptr{Void}}(C_NULL); nnz = Ref{Int64}(0)
    check(ccall((:mpb200_table_union_transpose, LIB), Cint, (Ptr{Void}, Ptr{Void}, Ref{Ptr{Void}}, Ref{Int64}), a, b, out, nnz))
    out[], nnz[]
end

# ---- GMT* on the device: mpb200_gmt_plan over tables and bits that never leave HBM ----------------------------
# C layouts of mpb200_gmt_desc / mpb200_gmt_result (include/mpb200.h).
immutable GmtDescC
    fwd::Ptr{Void}
    bwd::Ptr{Void}
    goal_bits::Ptr{UInt64}
    init::Int64
    width::Float64
    checkpts::Int32
    space::Ptr{SpaceDescC}
end
immutable GmtResultC
    solved::Int32
    grid_blocks::Int32
    goal::Int64
    cost::Float64
    iterations::Int64
    expansions::Int64
    checks::Int64
    checks_in_bounds::Int64
    path_len::Int64
end
"""gmtstar over device tables: s the sample set, tF / tB the forward / backward table handles (tB with its edge bits,
the same handle twice for a symmetric metric), goal a BitVector over the samples, w = lambda * r.  Points bits must have
been computed on s (mpb200_points_free) unless checkpts = false.  Returns (result, path, tree, costs)."""
function gmtstar_b200(s::B200Samples, tF::Ptr{Void}, tB::Ptr{Void}, goal::BitVector, w::Float64, sd::SpaceDesc;
                      checkpts = true)
    N = length(goal)
    path = Vector{Int64}(N); tree = Vector{Int64}(N); costs = Vector{Float64}(N)
    res = Ref{GmtResultC}()
    desc = Ref(GmtDescC(tF, tB, pointer(goal.chunks), 1, w, Int32(checkpts),
                        Base.unsafe_convert(Ptr{SpaceDescC}, sd.c)))        # goal and sd stay rooted by the arguments
    check(ccall((:mpb200_gmt_plan, LIB), Cint,
                (Ptr{Void}, Ref{GmtDescC}, Ref{GmtResultC}, Ptr{Int64}, Int64, Ptr{Int64}, Ptr{Float64}),
                s.h, desc, res, path, N, tree, costs))
    r = res[]
    r, path[1:r.path_len], tree, costs
end

# ---- PRM* on the device: mpb200_sssp_plan, the shortest path over the same tables and bits --------------------
# C layout of mpb200_sssp_result (include/mpb200.h); the descriptor is GmtDescC, whose width is ignored.
immutable SsspResultC
    solved::Int32
    grid_blocks::Int32
    goal::Int64
    cost::Float64
    path_len::Int64
    rounds::Int64
    levels::Int64
    reached::Int64
end
"""The roadmap-optimal plan (PRM*) over device tables, with the arguments of gmtstar_b200 but no width: the cheapest
path from sample 1 to the goal over every edge of tB whose bit is set.  tree and costs cover the vertices no costlier
than the goal (all reachable ones when the plan fails); the others have parent 0 and cost Inf.  Returns (result, path,
tree, costs)."""
function prmstar_b200(s::B200Samples, tF::Ptr{Void}, tB::Ptr{Void}, goal::BitVector, sd::SpaceDesc; checkpts = true)
    N = length(goal)
    path = Vector{Int64}(N); tree = Vector{Int64}(N); costs = Vector{Float64}(N)
    res = Ref{SsspResultC}()
    desc = Ref(GmtDescC(tF, tB, pointer(goal.chunks), 1, 0.0, Int32(checkpts),
                        Base.unsafe_convert(Ptr{SpaceDescC}, sd.c)))        # goal and sd stay rooted by the arguments
    check(ccall((:mpb200_sssp_plan, LIB), Cint,
                (Ptr{Void}, Ref{GmtDescC}, Ref{SsspResultC}, Ptr{Int64}, Int64, Ptr{Int64}, Ptr{Float64}),
                s.h, desc, res, path, N, tree, costs))
    r = res[]
    r, path[1:r.path_len], tree, costs
end
"""prmstar_b200 for a batch of queries over the same tables (mpb200_sssp_plan_batch): query q runs from sample
inits[q] to the goal mask goals[q], all in one device launch.  Each query's outputs equal those of its own
prmstar_b200 plan.  Returns, per query, (result, path, tree, costs).  Written out in full but not run: Julia is not
installed where this binding was written."""
function prmstar_batch_b200(s::B200Samples, tF::Ptr{Void}, tB::Ptr{Void}, inits::Vector{Int64},
                            goals::Vector{BitVector}, sd::SpaceDesc; checkpts = true)
    nq = length(inits); N = length(goals[1])
    descs = [GmtDescC(tF, tB, pointer(goals[q].chunks), inits[q], 0.0, Int32(checkpts),
                      Base.unsafe_convert(Ptr{SpaceDescC}, sd.c)) for q in 1:nq]   # goals and sd stay rooted
    res = Vector{SsspResultC}(nq)
    paths = Matrix{Int64}(N, nq); trees = Matrix{Int64}(N, nq); costs = Matrix{Float64}(N, nq)   # column q = query q
    check(ccall((:mpb200_sssp_plan_batch, LIB), Cint,
                (Ptr{Void}, Ptr{GmtDescC}, Int64, Ptr{SsspResultC}, Ptr{Int64}, Int64, Ptr{Int64}, Ptr{Float64}),
                s.h, descs, nq, res, paths, N, trees, costs))
    [(res[q], paths[1:res[q].path_len, q], trees[:, q], costs[:, q]) for q in 1:nq]
end

# C layout of mpb200_gmt_edges (include/mpb200.h): the motion check lazy GMT* runs on the one entry each candidate uses
const GMT_EDGES_STRAIGHT = Int32(0)
const GMT_EDGES_LQ = Int32(1)
const GMT_EDGES_CAR = Int32(2)
immutable GmtEdgesC
    kind::Int32
    obstacles::Ptr{Void}
    lq::Ptr{Void}
    r::Float64
    car_kind::Int32
    turning_radius::Float64
    speed::Float64
end
"""gmtstar_b200 without edge bits (mpb200_gmt_plan_lazy): the planning kernel runs is_free_motion(V[y], V[x]) itself on
the entry it would have looked up.  edges = GmtEdgesC(GMT_EDGES_STRAIGHT, obstacles, C_NULL, 0.0, 0, 0.0, 0.0), or
GMT_EDGES_LQ with the LQ handle and the steering horizon r, or GMT_EDGES_CAR with the car kind, turning radius and
speed.  tB needs no edge bits, and a new obstacle set replans over the same tables.  Returns (result, path, tree, costs,
segment tests run)."""
function gmtstar_lazy_b200(s::B200Samples, tF::Ptr{Void}, tB::Ptr{Void}, goal::BitVector, w::Float64, sd::SpaceDesc,
                           edges::GmtEdgesC; checkpts = true)
    N = length(goal)
    path = Vector{Int64}(N); tree = Vector{Int64}(N); costs = Vector{Float64}(N)
    res = Ref{GmtResultC}(); segs = Ref{Int64}(0)
    desc = Ref(GmtDescC(tF, tB, pointer(goal.chunks), 1, w, Int32(checkpts),
                        Base.unsafe_convert(Ptr{SpaceDescC}, sd.c)))
    check(ccall((:mpb200_gmt_plan_lazy, LIB), Cint,
                (Ptr{Void}, Ref{GmtDescC}, Ref{GmtEdgesC}, Ref{GmtResultC}, Ref{Int64}, Ptr{Int64}, Int64, Ptr{Int64},
                 Ptr{Float64}),
                s.h, desc, Ref(edges), res, segs, path, N, tree, costs))
    r = res[]
    r, path[1:r.path_len], tree, costs, segs[]
end

"""A batch of queries over one roadmap in one launch (mpb200_gmt_plan_batch): query q from sample inits[q] (1-based) to
goals[q] at width ws[q], over the tables and bits of gmtstar_b200 (edges === nothing) or with the motion check of
gmtstar_lazy_b200.  Each query's outputs equal that single call's for it.  Returns, per query, (result, path, tree,
costs, segment tests run).  Declared only: Julia is not installed where this binding was written, so it has not been
run."""
function gmtstar_batch_b200(s::B200Samples, tF::Ptr{Void}, tB::Ptr{Void}, inits::Vector{Int64}, goals::Vector{BitVector},
                            ws::Vector{Float64}, sd::SpaceDesc, edges::Union{GmtEdgesC, Void} = nothing;
                            checkpts = true)
    nq = length(inits); N = length(goals[1])
    descs = [GmtDescC(tF, tB, pointer(goals[q].chunks), inits[q], ws[q], Int32(checkpts),
                      Base.unsafe_convert(Ptr{SpaceDescC}, sd.c)) for q in 1:nq]   # goals and sd stay rooted
    res = Vector{GmtResultC}(nq); segs = zeros(Int64, nq)
    paths = Matrix{Int64}(N, nq); trees = Matrix{Int64}(N, nq); costs = Matrix{Float64}(N, nq)   # column q = query q
    check(ccall((:mpb200_gmt_plan_batch, LIB), Cint,
                (Ptr{Void}, Ptr{GmtDescC}, Int64, Ptr{GmtEdgesC}, Ptr{GmtResultC}, Ptr{Int64}, Ptr{Int64}, Int64,
                 Ptr{Int64}, Ptr{Float64}),
                s.h, descs, nq, edges === nothing ? C_NULL : Ref(edges), res, segs, paths, N, trees, costs))
    [(res[q], paths[1:res[q].path_len, q], trees[:, q], costs[:, q], segs[q]) for q in 1:nq]
end

# ---- shortcutting planned paths (mpb200_shortcut_paths; include/mpb200.h, DESIGN.md section 10c) -------------------
"""shortcut_paths_b200(paths, CC, sd; subdivisions = 4): for each path (a d x L matrix of states, e.g. statevec2mat of
a solution's states), the cheapest collision-free route through its subdivided waypoints under CC and the space of sd,
all paths in one device call.  Not the reference's shortcut / adaptive_shortcut! (postprocessors.jl): the cost is never
above the path's own, and a path that is not free comes back unchanged with cost Inf.  Returns, per path, (states as a
d x L' matrix, cost, pairs, segment tests run); the segment tests are added to CC.count.  Written out in full but not
run: Julia is not installed where this binding was written."""
function shortcut_paths_b200(paths::Vector{Matrix{Float64}}, CC::B200Checker, sd::SpaceDesc; subdivisions = 4)
    n = length(paths); d = size(paths[1], 1); k = Int32(subdivisions)
    offsets = zeros(Int64, n + 1)
    for q in 1:n
        offsets[q + 1] = offsets[q] + size(paths[q], 2)
    end
    Y = hcat(paths...)                                       # d x sum(L): AoS, path q at columns offsets[q]+1 ..
    cap = maximum((size(p, 2) - 1) * k + 1 for p in paths)
    out = Array(Float64, d, cap, n)                          # row q of the C layout = out[:, :, q]
    out_len = zeros(Int64, n); costs = zeros(Float64, n); pairs = zeros(Int64, n); segs = zeros(Int64, n)
    check(ccall((:mpb200_shortcut_paths, LIB), Cint,
                (Ptr{Float64}, Ptr{Int64}, Int64, Cint, Ptr{Void}, Ref{SpaceDescC}, Int32, Ptr{Float64}, Int64,
                 Ptr{Int64}, Ptr{Float64}, Ptr{Int64}, Ptr{Int64}),
                Y, offsets, n, d, CC.h, sd.c, k, out, cap, out_len, costs, pairs, segs))
    CC.count += sum(segs)
    [(out[:, 1:out_len[q], q], costs[q], pairs[q], segs[q]) for q in 1:n]
end

end # module
