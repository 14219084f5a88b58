# BeamletOpticsB200.jl -- reference-side binding of libbmo.so (the B200-native trace hot path).
#
# This is the file a BeamletOptics.jl maintainer would add (e.g. as a package extension): a new
# `CUDASystem <: AbstractSystem` whose `solve_system!` methods flatten `Leaves(system.objects)` into the
# plain tables of include/bmo.h and `ccall` the library.  Constructors, kinematics (`translate3d!`,
# `rotate3d!`, ...), `Beam` / `GaussianBeamlet` / `Photodetector` / `Spotdetector` stay the reference's
# own Julia objects; results land where the reference puts them (`pd.field`, `sd.data`, `beam.rays`).
#
# NOT EXERCISED IN THIS REPOSITORY: Julia is not installed in the build image.  The same ABI is driven
# and tested from Python (beamletoptics.jl_b200/_lib.py, flatten.py, solver.py); this file mirrors that
# code one to one.  Struct layouts below must match include/bmo.h (checked on the Python side by
# tests/test_abi.py::test_struct_layouts_match_header).
module BeamletOpticsB200

using BeamletOptics
using BeamletOptics: AbstractSystem, AbstractObject, AbstractSDF, AbstractMesh, UnionSDF, MeniscusLensSDF,
    PlanoSurfaceSDF, CylinderSDF, SphereSDF, ConvexSphericalSurfaceSDF, ConcaveSphericalSurfaceSDF,
    CutSphereSDF, BoxSDF, RingSDF, RightAnglePrismSDF, Mesh, Lens, Prism, DoubletLens, AbstractReflectiveOptic,
    ThinBeamsplitter, AbstractPlateBeamsplitter, CubeBeamsplitter, Photodetector, Spotdetector,
    IntersectableObject, NonInteractableObject, Beam, Ray, PolarizedRay, GaussianBeamlet, Intersection,
    position, orientation, transposed_orientation, shape, objects, refractive_index, wavelength, vertices, faces
using StaticArrays, GeometryBasics

const libbmo = get(ENV, "LIBBMO", "libbmo.so")

# ---- include/bmo.h, field for field ----------------------------------------------------------------
struct BmoPrim                      # bmo_prim
    type::Int32; reserved::Int32
    pos::NTuple{3,Float64}; tdir::NTuple{9,Float64}; par::NTuple{4,Float64}
    ext_first::Int32; ext_count::Int32          # aspheric / acylindric surfaces: parameter block in BmoTables.ext
end
struct BmoPart                      # bmo_part
    object::Int32; role::Int32; shape_kind::Int32; first::Int32; count::Int32; n_row::Int32
    reflectance::Float64; transmittance::Float64; bound::NTuple{10,Float64}   # sphere (centre, radius), box (lo, hi)
end
struct BmoObject                    # bmo_object
    kind::Int32; first_part::Int32; n_parts::Int32; pd_n::Int32
    pos::NTuple{3,Float64}; dir::NTuple{9,Float64}; pd_lo::Float64; pd_hi::Float64
end
struct BmoMesh                      # bmo_mesh
    first_vertex::Int64; n_vertices::Int64; first_face::Int64; n_faces::Int64; f32::Int32; reserved::Int32
end
struct BmoTables                    # bmo_tables
    n_prims::Int32;    prims::Ptr{BmoPrim}
    n_parts::Int32;    parts::Ptr{BmoPart}
    n_objects::Int32;  objects::Ptr{BmoObject}
    n_meshes::Int32;   meshes::Ptr{BmoMesh}
    n_vertices::Int64; vertices::Ptr{Float64}
    n_faces::Int64;    faces::Ptr{Int32}
    n_lambda::Int32;   lambdas::Ptr{Float64}
    n_rows::Int32;     n_table::Ptr{Float64}
    n_system::Float64
    n_ext::Int64;      ext::Ptr{Float64}        # c, k, d, max_sag[1], sag(d/2), sag'(d/2), n, coefficients... per aspheric primitive
    n_jones::Int32;    jones::Ptr{Float64}      # [n_jones][10]: GlobalJonesBasis (row-major) + cutoff of each PolarizationFilter
    norm_zero_rule::Int32; reserved::Int32
end
struct BmoResultInfo
    n_roots::Int64; n_beams::Int64; n_segments::Int64; interactions::Int64
    rays_per_beam::Int32; polarized::Int32; waves::Int32; reserved::Int32
end

const PRIM = Dict(PlanoSurfaceSDF => 0, CylinderSDF => 1, SphereSDF => 2, ConvexSphericalSurfaceSDF => 3,
    ConcaveSphericalSurfaceSDF => 4, CutSphereSDF => 5, BoxSDF => 6, RingSDF => 7, RightAnglePrismSDF => 8,
    BeamletOptics.ConvexCylinderSDF => 10, BeamletOptics.ConcaveCylinderSDF => 11)
const KEEP_SEGMENTS = UInt32(1)
const UNIFORM_DIR = UInt32(8)

check(rc) = rc == 0 || error(unsafe_string(ccall((:bmo_last_error, libbmo), Cstring, ())))

rowmajor(M) = ntuple(k -> Float64(M[(k - 1) ÷ 3 + 1, (k - 1) % 3 + 1]), 9)

# par[] per primitive type, exactly the fields each sdf(...) method reads (see bmo.h enum bmo_prim_type)
params(s::PlanoSurfaceSDF) = (s.thickness, s.diameter, 0.0, 0.0)
params(s::CylinderSDF) = (s.radius, s.height, 0.0, 0.0)
params(s::SphereSDF) = (s.radius, 0.0, 0.0, 0.0)
params(s::ConvexSphericalSurfaceSDF) = (s.radius, s.diameter, s.sag, s.height)
params(s::ConcaveSphericalSurfaceSDF) = (s.radius, s.diameter, s.sag, 0.0)
params(s::CutSphereSDF) = (s.radius, s.height, s.w, 0.0)
params(s::BoxSDF) = (s.x / 2, s.y / 2, s.z / 2, 0.0)          # half extents, as PrimitiveSDF.jl:41-46 uses them
params(s::RingSDF) = (s.inner_radius, s.hwidth, s.hthickness, 0.0)
params(s::RightAnglePrismSDF) = (s.x / 2, s.y / 2, s.z / 2, 0.0)

prim(s::AbstractSDF) = BmoPrim(PRIM[Base.typename(typeof(s)).wrapper], 0, Tuple(Float64.(position(s))),
    rowmajor(transposed_orientation(s)), Float64.(params(s)), 0, 0)
# cylindric surfaces (CylindricalSDF.jl): the constants each sdf call recomputes are passed precomputed
params(s::BeamletOptics.ConvexCylinderSDF) = (h = sqrt(s.radius^2 - (s.diameter / 2)^2); (s.radius, h, sqrt(s.radius^2 - h^2), s.height / 2))
params(s::BeamletOptics.ConcaveCylinderSDF) = (s.radius, s.diameter, s.height, BeamletOptics.sag(abs(s.radius), s.diameter))
# aspheric / acylindric surfaces: parameter block appended to `ext` (see include/bmo.h, BMO_PRIM_CONVEX_ASPH)
const ASPH = Dict(BeamletOptics.ConvexAsphericalSurfaceSDF => 12, BeamletOptics.ConcaveAsphericalSurfaceSDF => 13,
    BeamletOptics.AconvexCylinderSDF => 14, BeamletOptics.AconcaveCylinderSDF => 15)
function prim(s::Union{BeamletOptics.AbstractAsphericalSurfaceSDF,BeamletOptics.AbstractAcylindricalSurfaceSDF}, ext::Vector{Float64})
    c, k, d, α = 1 / s.radius, s.conic_constant, s.diameter, s.coefficients
    first = length(ext)
    append!(ext, (c, k, d, s.max_sag[1], BeamletOptics.aspheric_equation(d / 2, c, k, α),
        BeamletOptics.gradient_aspheric_equation(d / 2, c, k, α)[1], Float64(length(α)), α...))
    hx = s isa BeamletOptics.AbstractAcylindricalSurfaceSDF ? s.height / 2 : 0.0
    BmoPrim(ASPH[Base.typename(typeof(s)).wrapper], 0, Tuple(Float64.(position(s))), rowmajor(transposed_orientation(s)),
        (0.0, hx, 0.0, 0.0), first, length(ext) - first)
end

function emit_sdf!(prims, s::AbstractSDF, ext::Vector{Float64})
    first = length(prims)
    for m in (s isa UnionSDF ? s.sdfs : (s,))
        if m isa MeniscusLensSDF        # frame + children posed relative to it (MeniscusLensSDF.jl:42-46)
            push!(prims, BmoPrim(9, 0, Tuple(Float64.(position(m))), rowmajor(transposed_orientation(m)), (0.0, 0.0, 0.0, 0.0), 0, 0))
            push!(prims, prim(m.convex), prim(m.cylinder), prim(m.concave))
        else
            push!(prims, haskey(ASPH, Base.typename(typeof(m)).wrapper) ? prim(m, ext) : prim(m))
        end
    end
    return first, length(prims) - first
end

"""Wraps a reference `System`; `solve_system!` on it runs on the GPU."""
struct CUDASystem{S<:AbstractSystem} <: AbstractSystem
    system::S
    device::Int
end
CUDASystem(s::AbstractSystem) = CUDASystem(s, 0)
BeamletOptics.objects(cs::CUDASystem) = objects(cs.system)
BeamletOptics.refractive_index(cs::CUDASystem, λ) = refractive_index(cs.system, λ)

const CTX = Dict{Int,Ptr{Cvoid}}()
function context(dev)
    get!(CTX, dev) do
        h = Ref{Ptr{Cvoid}}(C_NULL)
        check(ccall((:bmo_init, libbmo), Int32, (Int32, Ref{Ptr{Cvoid}}), dev, h))
        h[]
    end
end

kind_of(o::DoubletLens) = (5, (o.front, o.back), (1, 2))
kind_of(o::CubeBeamsplitter) = (4, (o.front, o.back, o.coating), (1, 2, 4))
kind_of(o::AbstractPlateBeamsplitter) = (3, (o.substrate, o.coating), (3, 4))
kind_of(o::ThinBeamsplitter) = (2, (o,), (0,))
kind_of(o::AbstractReflectiveOptic) = (1, (o,), (0,))
kind_of(o::Photodetector) = (6, (o,), (0,))
kind_of(o::Spotdetector) = (7, (o,), (0,))
kind_of(o::BeamletOptics.PSFDetector) = (9, (o,), (0,))
kind_of(o::BeamletOptics.PolarizationFilter) = (10, (o,), (0,))
kind_of(o::IntersectableObject) = (8, (o,), (0,))
kind_of(o::AbstractObject) = (0, (o,), (0,))                 # Lens, Prism: AbstractRefractiveOptic

"""Leaves(system.objects) -> tables of include/bmo.h (same order: it is trace_all's tie-break order)."""
function flatten(cs::CUDASystem, λs::Vector{Float64}; norm_zero_rule = 1)
    prims, parts, objs, meshes = BmoPrim[], BmoPart[], BmoObject[], BmoMesh[]
    verts, fcs, ntab, owners, jones, ext = Float64[], Int32[], Float64[], Any[], Float64[], Float64[]
    leaves = [o for o in objects(cs) if !(o isa NonInteractableObject)]
    for (oi, o) in enumerate(leaves)
        kind, subs, roles = kind_of(o)
        sh0 = length(subs) == 1 ? shape(o) : nothing
        if o isa BeamletOptics.PolarizationFilter      # tables.jones row: J (3x3, row-major), cutoff
            J = BeamletOptics.static_data(o.JMat)
            append!(jones, (Float64(J[i, j]) for i in 1:3 for j in 1:3)); push!(jones, Float64(o.cutoff))
        end
        push!(objs, BmoObject(kind, length(parts), length(subs),
            o isa Photodetector ? length(o.x) : (o isa BeamletOptics.PolarizationFilter ? length(jones) ÷ 10 - 1 : 0),
            sh0 === nothing ? (0.0, 0.0, 0.0) : Tuple(Float64.(position(sh0))),
            sh0 === nothing ? ntuple(_ -> 0.0, 9) : rowmajor(orientation(sh0)),
            o isa Photodetector ? first(o.x) : 0.0, o isa Photodetector ? last(o.x) : 0.0))
        for (sub, role) in zip(subs, roles)
            sh = shape(sub)
            n_row = -1
            if hasmethod(refractive_index, Tuple{typeof(sub),Float64})
                n_row = length(ntab) ÷ length(λs)
                append!(ntab, (Float64(refractive_index(sub, λ)) for λ in λs))   # KeyError for an untabulated λ, like the reference
            end
            c, r = bounding_sphere(sh)
            rr = r * (1 + 1e-9) + 1e-6                  # the sphere's box is a valid (loose) box bound; flatten.py derives a tighter one
            bound = (c[1], c[2], c[3], rr, c[1] - rr, c[2] - rr, c[3] - rr, c[1] + rr, c[2] + rr, c[3] + rr)
            R = sub isa ThinBeamsplitter ? (sub.reflectance, sub.transmittance) : (0.0, 0.0)
            if sh isa AbstractSDF
                first, count = emit_sdf!(prims, sh, ext)
                push!(parts, BmoPart(oi - 1, role, 0, first, count, n_row, R[1], R[2], bound))
            else
                V, F = vertices(sh), faces(sh)
                push!(meshes, BmoMesh(length(verts) ÷ 3, size(V, 1), length(fcs) ÷ 3, size(F, 1), eltype(V) == Float32 ? 1 : 0, 0))
                push!(parts, BmoPart(oi - 1, role, 1, length(meshes) - 1, 1, n_row, R[1], R[2], bound))
                append!(verts, Float64.(permutedims(V)))          # xyz triples; Float32 values widened, not rescaled
                append!(fcs, Int32.(permutedims(F) .- 1))
            end
            push!(owners, sub)
        end
    end
    return (; prims, parts, objs, meshes, verts, fcs, ntab, owners, leaves, λs, norm_zero_rule, jones, ext)
end

# conservative world-space bounding sphere of a shape (only used for result-identical early exits)
function bounding_sphere(sh::AbstractMesh)
    V = vertices(sh); c = vec(sum(V, dims = 1)) ./ size(V, 1)
    return c, maximum(norm(V[i, :] .- c) for i in 1:size(V, 1))
end
function bounding_sphere(sh::AbstractSDF)
    # half of a generous axis-aligned extent in the local frame, see shapes.py:local_bound for the per-type radii
    ms = sh isa UnionSDF ? sh.sdfs : (sh,)
    c = sum(Float64.(position(m)) for m in ms) ./ length(ms)
    return c, maximum(norm(Float64.(position(m)) .- c) + local_radius(m) for m in ms)
end
local_radius(s::PlanoSurfaceSDF) = hypot(s.diameter / 2, s.thickness)
local_radius(s::CylinderSDF) = hypot(s.radius, s.height)
local_radius(s::SphereSDF) = s.radius
local_radius(s::ConvexSphericalSurfaceSDF) = hypot(s.diameter / 2, s.sag)
local_radius(s::ConcaveSphericalSurfaceSDF) = hypot(s.diameter / 2, s.sag)
local_radius(s::CutSphereSDF) = s.radius
local_radius(s::BoxSDF) = norm((s.x, s.y, s.z)) / 2
local_radius(s::RingSDF) = hypot(s.inner_radius + s.hwidth, s.hthickness)
local_radius(s::RightAnglePrismSDF) = norm((s.x, s.y, s.z)) / 2
local_radius(s::MeniscusLensSDF) = maximum(norm(position(c)) + local_radius(c) for c in (s.convex, s.cylinder, s.concave))
# cylindric, aspheric and acylindric lens surfaces: generous radii (the flattener only needs a bound, shapes.py:local_bound is tighter)
local_radius(s::Union{BeamletOptics.ConvexCylinderSDF,BeamletOptics.ConcaveCylinderSDF}) = hypot(s.height / 2, s.diameter / 2) + s.diameter
local_radius(s::BeamletOptics.AbstractAsphericalSurfaceSDF) = hypot(s.diameter / 2, maximum(abs, s.max_sag)) + s.diameter / 2
local_radius(s::BeamletOptics.AbstractAcylindricalSurfaceSDF) = hypot(s.height / 2, s.diameter / 2, maximum(abs, s.max_sag)) + s.diameter / 2
local_radius(s::AbstractSDF) = error("BeamletOpticsB200: no bounding radius for $(typeof(s)) -- this SDF type is not supported by the GPU path")

function upload_tables(cs::CUDASystem, f)
    sys = Ref{Ptr{Cvoid}}(C_NULL)
    GC.@preserve f begin
        t = BmoTables(length(f.prims), pointer(f.prims), length(f.parts), pointer(f.parts), length(f.objs), pointer(f.objs),
            length(f.meshes), pointer(f.meshes), length(f.verts) ÷ 3, pointer(f.verts), length(f.fcs) ÷ 3, pointer(f.fcs),
            length(f.λs), pointer(f.λs), length(f.ntab) ÷ length(f.λs), pointer(f.ntab), 1.0,
            length(f.ext), pointer(f.ext), length(f.jones) ÷ 10, pointer(f.jones), f.norm_zero_rule, 0)
        check(ccall((:bmo_system_upload, libbmo), Int32, (Ptr{Cvoid}, Ref{BmoTables}, Ref{Ptr{Cvoid}}), context(cs.device), t, sys))
    end
    return sys[]
end

# One uploaded copy per CUDASystem, reused while the flattened tables do not change (solver.py: cached_system): poses are static
# during a solve and usually between the solves of a loop as well; the BVH of an STL mesh is built at upload, so re-uploading an
# unchanged system on every solve_system! would rebuild it every time.  Moving an object changes the hash and triggers an upload.
const UPLOADED = IdDict{Any,Tuple{UInt64,Ptr{Cvoid}}}()
tables_hash(f) = hash((f.prims, f.parts, f.objs, f.meshes, f.verts, f.fcs, f.ntab, f.λs, f.jones, f.ext, f.norm_zero_rule))
function upload(cs::CUDASystem, f)
    h = tables_hash(f)
    hit = get(UPLOADED, cs.system, nothing)
    hit !== nothing && hit[1] == h && return hit[2]
    hit !== nothing && ccall((:bmo_system_free, libbmo), Int32, (Ptr{Cvoid},), hit[2])
    sys = upload_tables(cs, f)
    UPLOADED[cs.system] = (h, sys)
    return sys
end
"""Hand the device memory the library keeps for reuse (parked blocks, its share of the stream-ordered pool) back to the driver."""
trim!(device::Integer = 0) = (n = Ref{Int64}(0); check(ccall((:bmo_trim, libbmo), Int32, (Ptr{Cvoid}, Ref{Int64}), context(device), n)); n[])

"""Release the device copy of a system (the cache otherwise keeps it until the next upload of a changed system)."""
function release!(cs::CUDASystem)
    hit = pop!(UPLOADED, cs.system, nothing)
    hit === nothing || ccall((:bmo_system_free, libbmo), Int32, (Ptr{Cvoid},), hit[2])
    return cs
end

"""
    solve_system!(cs::CUDASystem, beams::AbstractVector{<:Beam}; r_max = 100, retrace = true)

Replaces the serial loop of `src/System.jl:463-468`: all beams are traced in one call of
`bmo_trace_rays`; `Spotdetector.data` receives the hits in ray order, and each `Beam` gets its
segments back (`rays`, `children`) unless `rebuild = false` (throughput runs).
"""
function BeamletOptics.solve_system!(cs::CUDASystem, beams::AbstractVector{<:Beam{T,R}}; r_max = 100, retrace = true, rebuild = true) where {T,R}
    λs = unique(Float64(wavelength(first(b.rays))) for b in beams)
    f = flatten(cs, λs); sys = upload(cs, f)
    n = length(beams)
    pos = Matrix{Float64}(undef, 3, n); dir = similar(pos); lam = Vector{Int32}(undef, n)
    E0 = R <: PolarizedRay ? Matrix{Float64}(undef, 6, n) : nothing
    for (i, b) in enumerate(beams)
        r = first(b.rays)
        pos[:, i] .= position(r); dir[:, i] .= BeamletOptics.direction(r); lam[i] = findfirst(==(Float64(wavelength(r))), λs) - 1
        E0 === nothing || (E0[:, i] .= reinterpret(Float64, collect(ComplexF64.(r.E0))))
    end
    res = Ref{Ptr{Cvoid}}(C_NULL)
    prev = retrace ? get(SOLUTIONS, first(beams), C_NULL) : C_NULL     # the stored solution of these beams, if any
    if prev != C_NULL
        # retrace_system! (System.jl:188-255) for every beam of the stored trees, then solve_leaf!
        check(ccall((:bmo_retrace, libbmo), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Int32, UInt32, Ref{Ptr{Cvoid}}), sys, prev, r_max, KEEP_SEGMENTS, res))
        ccall((:bmo_result_free, libbmo), Int32, (Ptr{Cvoid},), prev)
    else
        GC.@preserve pos dir lam E0 begin
            # a collimated bundle ships its one direction once (BMO_UNIFORM_DIR: 24 B per ray over the bus instead of 48)
            flags = (rebuild ? KEEP_SEGMENTS : UInt32(0)) | (all(c -> c == view(dir, :, 1), eachcol(dir)) ? UNIFORM_DIR : UInt32(0))
            check(ccall((:bmo_trace_rays, libbmo), Int32,
                (Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Ptr{Float64}, Ptr{Int32}, Int32, UInt32, Ref{Ptr{Cvoid}}),
                sys, n, pos, dir, lam, E0 === nothing ? C_NULL : pointer(E0), C_NULL, r_max, flags, res))
        end
    end
    collect_spots!(f, res[])
    collect_psfs!(f, sys, res[])
    rebuild && rebuild_beams!(beams, f, res[])
    if rebuild
        SOLUTIONS[first(beams)] = res[]                # kept on the device for the next solve_system!(...; retrace = true)
    else
        ccall((:bmo_result_free, libbmo), Int32, (Ptr{Cvoid},), res[])
    end
    return nothing
end
BeamletOptics.solve_system!(cs::CUDASystem, bg::BeamletOptics.AbstractBeamGroup; kw...) = BeamletOptics.solve_system!(cs, BeamletOptics.beams(bg); kw...)
BeamletOptics.solve_system!(cs::CUDASystem, b::Beam; kw...) = BeamletOptics.solve_system!(cs, [b]; kw...)

"""GaussianBeamlets: `bmo_trace_beamlets`, then `bmo_pd_accumulate` adds into every `Photodetector.field` and
`bmo_psf_collect` appends to every `PSFDetector`."""
function BeamletOptics.solve_system!(cs::CUDASystem, gs::AbstractVector{<:GaussianBeamlet}; r_max = 100, retrace = true)
    λs = unique(Float64(g.λ) for g in gs)
    f = flatten(cs, λs); sys = upload(cs, f)
    n = length(gs)
    rays = Array{Float64}(undef, 6, 3, n)          # [pos; dir] x (chief, waist, divergence) x beamlet
    for (i, g) in enumerate(gs), (k, b) in enumerate((g.chief, g.waist, g.divergence))
        r = first(b.rays); rays[1:3, k, i] .= position(r); rays[4:6, k, i] .= BeamletOptics.direction(r)
    end
    lam = Int32[findfirst(==(Float64(g.λ)), λs) - 1 for g in gs]
    w0 = Float64[g.w0 for g in gs]; E0 = ComplexF64[g.E0 for g in gs]
    res = Ref{Ptr{Cvoid}}(C_NULL)
    GC.@preserve rays lam w0 E0 begin
        check(ccall((:bmo_trace_beamlets, libbmo), Int32,
            (Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Int32}, Ptr{Float64}, Ptr{ComplexF64}, Ptr{Int32}, Int32, UInt32, Ref{Ptr{Cvoid}}),
            sys, n, rays, lam, w0, E0, C_NULL, r_max, UInt32(0), res))
    end
    for (oi, o) in enumerate(f.leaves)
        o isa Photodetector || continue
        fld = o.field                                # Matrix{ComplexF64}, column-major [i, j]: exactly the ABI's layout
        GC.@preserve fld check(ccall((:bmo_pd_accumulate, libbmo), Int32,
            (Ptr{Cvoid}, Ptr{Cvoid}, Int32, Int32, Ptr{ComplexF64}, UInt32), sys, res[], oi - 1, 0, fld, UInt32(0)))
    end
    collect_spots!(f, res[])
    collect_psfs!(f, sys, res[])                     # three records per beamlet: chief, waist, divergence
    rebuild_beamlets!(gs, f, res[])
    ccall((:bmo_result_free, libbmo), Int32, (Ptr{Cvoid},), res[])
    return nothing
end
BeamletOptics.solve_system!(cs::CUDASystem, g::GaussianBeamlet; kw...) = BeamletOptics.solve_system!(cs, [g]; kw...)

# Stored solutions (bmo_result with its segment table), keyed by the first beam of the solved vector; the
# reference keeps the same information inside the Beam objects (rays, intersections, children).
const SOLUTIONS = IdDict{Any,Ptr{Cvoid}}()

# PSFDetector: the detector's `data` lives on the device (bmo_psf), keyed by the detector object
const PSFS = IdDict{Any,Tuple{Ptr{Cvoid},Any,Int}}()
function collect_psfs!(f, sys, res)
    for (oi, o) in enumerate(f.leaves)
        o isa BeamletOptics.PSFDetector || continue
        h = Ref{Ptr{Cvoid}}(haskey(PSFS, o) ? PSFS[o][1] : C_NULL); n = Ref{Int64}(0)
        check(ccall((:bmo_psf_collect, libbmo), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Int32, Ref{Ptr{Cvoid}}, Ref{Int64}), sys, res, oi - 1, h, n))
        PSFS[o] = (h[], f, oi - 1)
    end
end
"""intensity(psf; n, crop_factor, center, ...) (PSFDetector.jl:190-237) on the GPU: `bmo_psf_lims` + `bmo_psf_intensity`."""
function gpu_intensity(cs::CUDASystem, psf::BeamletOptics.PSFDetector; n = 100, crop_factor = 1, center = :centroid,
        x_min = Inf, x_max = Inf, z_min = Inf, z_max = Inf, x0_shift = 0.0, z0_shift = 0.0)
    h, f, oi = PSFS[psf]
    sys = upload(cs, flatten(cs, f.λs))
    lims = zeros(4)
    check(ccall((:bmo_psf_lims, libbmo), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Int32, Int32, Float64, Int32, Ptr{Float64}),
        sys, h, oi, 0, crop_factor, center == :centroid ? 0 : 1, lims))
    x_min != Inf && x_max != Inf && (lims[1] = x_min; lims[2] = x_max)
    z_min != Inf && z_max != Inf && (lims[3] = z_min; lims[4] = z_max)
    I = Matrix{Float64}(undef, n, n)
    check(ccall((:bmo_psf_intensity, libbmo), Int32,
        (Ptr{Cvoid}, Ptr{Cvoid}, Int32, Int32, Int32, Ptr{Float64}, Float64, Float64, Ptr{Float64}, UInt32),
        sys, h, oi, 0, n, lims, x0_shift, z0_shift, I, UInt32(0)))
    return LinRange(lims[1], lims[2], n) .+ x0_shift, LinRange(lims[3], lims[4], n) .+ z0_shift, I
end
function Base.empty!(psf::BeamletOptics.PSFDetector, ::Type{CUDASystem})
    haskey(PSFS, psf) && (ccall((:bmo_psf_free, libbmo), Int32, (Ptr{Cvoid},), PSFS[psf][1]); delete!(PSFS, psf))
    return psf
end

function info(res)
    i = Ref(BmoResultInfo(0, 0, 0, 0, 0, 0, 0, 0))
    check(ccall((:bmo_result_get_info, libbmo), Int32, (Ptr{Cvoid}, Ref{BmoResultInfo}), res, i)); i[]
end

"""Per-beam tables of a result: parent, child slot, nseg, status, first segment row, (Gaussian) w0 and E0."""
function beam_tables(res)
    nfo = info(res); nb = nfo.n_beams
    parent = Vector{Int32}(undef, nb); slot = similar(parent); nseg = similar(parent); status = similar(parent)
    first_seg = Vector{Int64}(undef, nb); w0 = Vector{Float64}(undef, nb); E0 = Vector{ComplexF64}(undef, nb)
    gauss = nfo.rays_per_beam == 3
    check(ccall((:bmo_result_beams, libbmo), Int32,
        (Ptr{Cvoid}, Ptr{Int32}, Ptr{Int32}, Ptr{Int32}, Ptr{Int32}, Ptr{Int64}, Ptr{Float64}, Ptr{ComplexF64}, Ptr{Int32}),
        res, parent, slot, nseg, status, first_seg, gauss ? pointer(w0) : C_NULL, gauss ? pointer(E0) : C_NULL, C_NULL))
    return (; nfo, nb, parent, slot, nseg, status, first_seg, w0, E0)
end

"""Beam ids in the reference's processing order (System.jl:444-461): root by root, each tree level by level, children as
[transmitted, reflected] -- the order in which `interact3d(::Spotdetector, ...)` pushes its hits (solver.py: bfs_order)."""
function bfs_order(bt)
    nb, nroots = bt.nb, bt.nfo.n_roots
    nb == nroots && return collect(1:nb)
    root = collect(1:nb); depth = zeros(Int, nb); code = zeros(Int, nb)
    for i in nroots+1:nb                       # children always have larger ids than their parent
        p = bt.parent[i] + 1
        root[i], depth[i], code[i] = root[p], depth[p] + 1, 2 * code[p] + bt.slot[i]
    end
    return sortperm(collect(zip(root, depth, code)))
end

function collect_spots!(f, res)
    bt = beam_tables(res); R = bt.nfo.rays_per_beam; n = bt.nb * R
    obj = Vector{Int32}(undef, n); xz = Matrix{Float64}(undef, 2, n)
    check(ccall((:bmo_result_spots, libbmo), Int32, (Ptr{Cvoid}, Ptr{Int32}, Ptr{Float64}), res, obj, xz))
    for b in bfs_order(bt), r in 1:R
        i = (b - 1) * R + r
        obj[i] >= 0 && push!(f.leaves[obj[i] + 1].data, Point2(xz[1, i], xz[2, i]))      # Spotdetector.jl:50-61
    end
end

"""Segment table of a result as column arrays (rows = n_segments * rays_per_beam; Gaussian: chief, waist, divergence interleaved)."""
function segment_tables(res, nfo)
    ns = nfo.n_segments * nfo.rays_per_beam
    pos = Matrix{Float64}(undef, 3, ns); dir = similar(pos); nrm = similar(pos)
    n = Vector{Float64}(undef, ns); t = similar(n); obj = Vector{Int32}(undef, ns); part = similar(obj)
    E0 = nfo.polarized != 0 ? Matrix{ComplexF64}(undef, 3, ns) : nothing
    check(ccall((:bmo_result_segments, libbmo), Int32,
        (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Ptr{Int32}, Ptr{ComplexF64}),
        res, pos, dir, n, t, nrm, obj, part, E0 === nothing ? C_NULL : pointer(E0)))
    return (; pos, dir, nrm, n, t, obj, part, E0)
end

# one ray of the segment table as the reference's mutable struct (Rays.jl:14-20, PolarizedRays.jl:37-44); the stored direction
# is the tracer's (refracted directions are not re-normalised, Lenses.jl:69), so the fields are set directly
function make_ray(::Type{Ray{T}}, sg, s, λ, f) where {T}
    Ray{T}(Point3{T}(sg.pos[:, s]), Point3{T}(sg.dir[:, s]), make_intersection(T, sg, s, f), T(λ), T(sg.n[s]))
end
function make_ray(::Type{PolarizedRay{T}}, sg, s, λ, f) where {T}
    PolarizedRay{T}(Point3{T}(sg.pos[:, s]), Point3{T}(sg.dir[:, s]), make_intersection(T, sg, s, f), T(λ), T(sg.n[s]),
        Point3{Complex{T}}(sg.E0[:, s]))
end
# t = Inf <=> intersection === nothing (AbstractRay.jl:13-18: fields object, shape, t, n)
make_intersection(::Type{T}, sg, s, f) where {T} = isfinite(sg.t[s]) ?
    Intersection{T}(f.leaves[sg.obj[s] + 1], shape(f.owners[sg.part[s] + 1]), T(sg.t[s]), Point3{T}(sg.nrm[:, s])) : nothing

# Beam trees from the segment table (Beam.jl:13-79): roots keep their identity, children are created in id order (a child's id
# is larger than its parent's; slot 0 = transmitted is numbered before slot 1 = reflected, which is the push! order of
# ThinBeamsplitter.jl:150-168)
function rebuild_beams!(beams::AbstractVector{<:Beam{T,R}}, f, res) where {T,R}
    bt = beam_tables(res); sg = segment_tables(res, bt.nfo)
    made = Vector{Beam{T,R}}(undef, bt.nb)
    for b in 1:bt.nb
        root = b <= length(beams)
        λ = wavelength(first((root ? beams[b] : made[bt.parent[b] + 1]).rays))
        rays = R[make_ray(R, sg, s, λ, f) for s in bt.first_seg[b] + 1:bt.first_seg[b] + bt.nseg[b]]
        if root
            beams[b].rays = rays; empty!(beams[b].children); made[b] = beams[b]
        else
            p = made[bt.parent[b] + 1]
            made[b] = Beam{T,R}(rays, p, Vector{Beam{T,R}}())
            push!(p.children, made[b])
        end
    end
end

# GaussianBeamlet trees (Gaussian.jl:33-42, 96-111): three Beam{T,Ray{T}} per beamlet whose rays are rows 3k+1 (chief),
# 3k+2 (waist), 3k+3 (divergence) of the segment table; children carry the w0 / E0 the splitter gave them
# (ThinBeamsplitter.jl:104-148) and are linked with parent! (child.chief.parent = parent.chief, needed by length / point_on_beam)
function rebuild_beamlets!(gs::AbstractVector{GaussianBeamlet{T}}, f, res) where {T}
    bt = beam_tables(res); sg = segment_tables(res, bt.nfo)
    made = Vector{GaussianBeamlet{T}}(undef, bt.nb)
    RT = Ray{T}
    for b in 1:bt.nb
        root = b <= length(gs)
        λ = root ? gs[b].λ : made[bt.parent[b] + 1].λ
        rows = bt.first_seg[b] .+ (0:bt.nseg[b] - 1)
        three = ntuple(k -> RT[make_ray(RT, sg, 3 * r + k, λ, f) for r in rows], 3)
        if root
            g = gs[b]
            g.chief.rays, g.waist.rays, g.divergence.rays = three
            empty!(g.children); empty!(g.chief.children); empty!(g.waist.children); empty!(g.divergence.children)
            made[b] = g
        else
            p = made[bt.parent[b] + 1]
            mk(rays) = Beam{T,RT}(rays, nothing, Vector{Beam{T,RT}}())
            g = GaussianBeamlet(mk(three[1]), mk(three[2]), mk(three[3]), T(λ), T(bt.w0[b]), Complex{T}(bt.E0[b]))
            BeamletOptics.parent!(g, p)
            push!(p.children, g)
            made[b] = g
        end
    end
end

# ---- multi-GPU: one process per GPU (Distributed / MPI.jl / a shared file carry the 128-byte id) -----------------------
"""`id = comm_unique_id()` on rank 0, shipped to every rank, then `comm = comm_init(cs, n_ranks, rank, id)` on all of them."""
function comm_unique_id()
    id = Vector{UInt8}(undef, 128)
    check(ccall((:bmo_comm_unique_id, libbmo), Int32, (Ptr{UInt8},), id)); id
end
function comm_init(cs::CUDASystem, n_ranks::Integer, rank::Integer, id::Vector{UInt8})
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:bmo_comm_init, libbmo), Int32, (Ptr{Cvoid}, Int32, Int32, Ptr{UInt8}, Ref{Ptr{Cvoid}}), context(cs.device), n_ranks, rank, id, h)); h[]
end
"""Sum the ranks' partial `pd.field`s in place (bmo_pd_allreduce: NCCL inside libbmo.so) after each rank solved its share of the beamlets."""
allreduce_field!(comm, pd::Photodetector) = (fld = pd.field; GC.@preserve fld check(ccall((:bmo_pd_allreduce, libbmo), Int32,
    (Ptr{Cvoid}, Ptr{ComplexF64}, Int64, UInt32), comm, fld, length(fld), UInt32(0))); pd)
comm_free(comm) = ccall((:bmo_comm_free, libbmo), Int32, (Ptr{Cvoid},), comm)

end # module
