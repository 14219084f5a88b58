/* bmo.h -- C ABI of libbmo.so, the B200-native (sm_100a) trace hot path behind BeamletOptics.jl's
 * solve_system! seam.
 *
 * The reference (pure Julia, /root/reference) has no FFI boundary; its extension mechanism is
 * multiple dispatch on `solve_system!(system::AbstractSystem, beam; r_max, retrace)`
 * (src/System.jl:444-468).  A host-side `CUDASystem <: AbstractSystem` (Julia, see INTEGRATION.md)
 * or the Python mirror in beamletoptics.jl_b200/ flattens `Leaves(system.objects)`
 * (src/System.jl:21) into the plain tables below and calls these entry points via ccall/ctypes.
 * All functions return 0 on success or a negative BMO_E* code; bmo_last_error() gives the text.
 * No exceptions cross the boundary, no torch/Julia types appear in signatures, the caller owns
 * every input array and every output buffer it passes in.
 *
 * All arithmetic is FP64 (complex128 for fields / Jones vectors).
 */
#ifndef BMO_H
#define BMO_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BMO_OK 0
#define BMO_EINVAL (-1)   /* bad argument (reference: ArgumentError / ErrorException) */
#define BMO_ECUDA (-2)    /* CUDA runtime error */
#define BMO_ENOMEM (-3)
#define BMO_ESTATE (-4)   /* call order / handle misuse */
#define BMO_ENCCL (-5)    /* NCCL missing (dlopen failed) or an NCCL call failed */

/* ---- SDF primitives: replaces the `sdf(shape, point)` methods of
 * src/SDFs/SphericalLensSDF.jl:60-65,86-89,159-170,219-232, src/SDFs/PrimitiveSDF.jl:41-46,71-76,
 * 112-124,162-166,204-210 and src/SDFs/MeniscusLensSDF.jl:42-46.  par[] per type:               */
enum bmo_prim_type {
    BMO_PRIM_PLANO = 0,     /* par: thickness, diameter                          */
    BMO_PRIM_CYLINDER = 1,  /* par: radius, half height                          */
    BMO_PRIM_SPHERE = 2,    /* par: radius                                       */
    BMO_PRIM_CONVEX = 3,    /* par: radius, diameter, sag, height                */
    BMO_PRIM_CONCAVE = 4,   /* par: radius, diameter, sag                        */
    BMO_PRIM_CUTSPHERE = 5, /* par: radius, height, w                            */
    BMO_PRIM_BOX = 6,       /* par: half extents x, y, z                         */
    BMO_PRIM_RING = 7,      /* par: inner_radius(+hwidth), hwidth, hthickness    */
    BMO_PRIM_RAPRISM = 8,   /* par: half extents x, y, z                         */
    BMO_PRIM_CONVEX_CYL = 10, /* ConvexCylinderSDF (CylindricalSDF.jl:30-78); par: radius, cut height sqrt(r^2-(d/2)^2),
                                 w = sqrt(r^2 - cut height^2), half extrusion height                  */
    BMO_PRIM_CONCAVE_CYL = 11,/* ConcaveCylinderSDF (CylindricalSDF.jl:92-133); par: radius (signed), diameter, height,
                                 sag(|radius|, diameter)                                            */
    BMO_PRIM_CONVEX_ASPH = 12,/* ConvexAsphericalSurfaceSDF (AsphericalLensSDF.jl:22-31, 188-240, 309-328): parameters in
                                 tables.ext[ext_first ...]: c = 1/radius, conic constant, diameter, max_sag[1],
                                 aspheric_equation(d/2), gradient_aspheric_equation(d/2)[1], n coefficients, coefficients.
                                 Normals by central differences only (:3-5).                        */
    BMO_PRIM_CONCAVE_ASPH = 13,/* ConcaveAsphericalSurfaceSDF (:88-98, 242-307, 330-349), same parameter block */
    BMO_PRIM_CONVEX_ACYL = 14,/* AconvexCylinderSDF (AcylindricalSDF.jl:14-72): the aspheric profile in (z, y) extruded along x;
                                 parameter block as for the aspheres, par[1] = half extrusion height; AD normals */
    BMO_PRIM_CONCAVE_ACYL = 15,/* AconcaveCylinderSDF (:74-120)                                     */
    BMO_PRIM_MENISCUS = 9   /* frame only; followed by 3 child records: convex, cylinder, concave,
                               posed relative to this frame (MeniscusLensSDF.jl:42-46)            */
};
typedef struct bmo_prim {
    int32_t type;
    int32_t reserved;
    double pos[3];   /* position(shape)                                   (AbstractSDF.jl:35-40) */
    double tdir[9];  /* transposed_orientation(shape), row-major: local = tdir * (P - pos)       */
    double par[4];
    int32_t ext_first;   /* aspheric surfaces: first double of the parameter block in tables.ext, else 0        */
    int32_t ext_count;   /* length of that block                                                             */
} bmo_prim;

/* ---- parts: one shape each.  A part is what `shape(intersection)` / `Hint.shape` identify
 * (src/AbstractTypes/AbstractRay.jl:13-18, AbstractSystem.jl:49-57).                             */
enum bmo_shape_kind { BMO_SHAPE_SDF = 0, BMO_SHAPE_MESH = 1 };
enum bmo_role {
    BMO_ROLE_SINGLE = 0,     /* SingleShape object                                                */
    BMO_ROLE_FRONT = 1,      /* DoubletLens.front / CubeBeamsplitter.front                        */
    BMO_ROLE_BACK = 2,       /* DoubletLens.back  / CubeBeamsplitter.back                         */
    BMO_ROLE_SUBSTRATE = 3,  /* AbstractPlateBeamsplitter.substrate                               */
    BMO_ROLE_COATING = 4     /* ThinBeamsplitter coating of a plate / cube splitter               */
};
typedef struct bmo_part {
    int32_t object;      /* owning object (index into objects)                                    */
    int32_t role;
    int32_t shape_kind;
    int32_t first;       /* SDF: first prim record; MESH: mesh index                              */
    int32_t count;       /* SDF: number of prim records of the union (meniscus children included) */
    int32_t n_row;       /* row of n_table for refractive parts, else -1                          */
    double reflectance;  /* coating amplitudes sqrt(R), sqrt(1-R^2)  (ThinBeamsplitter.jl:43-51)   */
    double transmittance;
    double bound[10];    /* conservative world-space bounds of the part: sphere (centre xyz, radius) and
                            axis-aligned box (lo xyz, hi xyz), both inflated; only used for
                            result-identical early exits (guaranteed misses, parts that cannot beat
                            the closest hit found so far)                                         */
} bmo_part;

/* ---- objects in `Leaves(system.objects)` order (tie-break order of trace_all, System.jl:57-72).
 * NonInteractableObject is skipped by the flattener (NonInteractable.jl:19-20).                  */
enum bmo_obj_kind {
    BMO_OBJ_REFRACTIVE = 0,   /* Lens, Prism            (Lenses.jl:46-126)                        */
    BMO_OBJ_MIRROR = 1,       /* AbstractReflectiveOptic (Mirrors.jl:39-69)                       */
    BMO_OBJ_THIN_BS = 2,      /* ThinBeamsplitter       (ThinBeamsplitter.jl:108-168)             */
    BMO_OBJ_PLATE_BS = 3,     /* parts: substrate, coating (PlateBeamsplitter.jl:160-275)         */
    BMO_OBJ_CUBE_BS = 4,      /* parts: front, back, coating (CubeBeamsplitter.jl:63-121)         */
    BMO_OBJ_DOUBLET = 5,      /* parts: front, back     (DoubletLenses.jl:66-76)                  */
    BMO_OBJ_PHOTODETECTOR = 6,/* (Photodetector.jl:69-107)                                        */
    BMO_OBJ_SPOTDETECTOR = 7, /* (Spotdetector.jl:50-61)                                          */
    BMO_OBJ_STOP = 8,         /* IntersectableObject    (Intersectable.jl:15)                     */
    BMO_OBJ_POLFILTER = 10,   /* PolarizationFilter     (Polarizers/PolarizationFilter.jl:31-47, JonesCalculus.jl:29-46):
                                 pd_n = row of tables.jones; orientation(object) = dir                 */
    BMO_OBJ_PSFDETECTOR = 9   /* PSFDetector            (Detectors/PSFDetector.jl:77-89): absorbs; the hit records are
                                 rebuilt from the segment table by bmo_psf_collect                */
};
typedef struct bmo_object {
    int32_t kind;
    int32_t first_part;
    int32_t n_parts;
    int32_t pd_n;        /* Photodetector: pixels per side                                        */
    double pos[3];       /* detectors: position(shape)                                            */
    double dir[9];       /* detectors: orientation(shape), row-major                              */
    double pd_lo, pd_hi; /* Photodetector: x = y = LinRange(pd_lo, pd_hi, pd_n) (Photodetector.jl:52) */
} bmo_object;

typedef struct bmo_mesh {
    int64_t first_vertex, n_vertices;  /* into vertices[] (xyz triples, WORLD coordinates, Mesh.jl:33-39) */
    int64_t first_face, n_faces;       /* into faces[] (3 x int32 each, 0-based, mesh-local vertex ids)   */
    int32_t f32;                       /* 1: Mesh{Float32} (STL, Mesh.jl:48-70): edge vectors and face normals
                                          are formed in Float32 like the reference's Point3{Float32} arithmetic */
    int32_t reserved;
} bmo_mesh;

typedef struct bmo_tables {
    int32_t n_prims;    const bmo_prim* prims;
    int32_t n_parts;    const bmo_part* parts;
    int32_t n_objects;  const bmo_object* objects;
    int32_t n_meshes;   const bmo_mesh* meshes;
    int64_t n_vertices; const double* vertices;
    int64_t n_faces;    const int32_t* faces;
    int32_t n_lambda;   const double* lambdas;   /* distinct vacuum wavelengths of the beams       */
    int32_t n_rows;     const double* n_table;   /* [n_rows][n_lambda] refractive_index(obj, lambda),
                                                    evaluated on the host (Lenses.jl:37-38)        */
    double n_system;                             /* refractive_index(system, lambda) = 1.0 (AbstractSystem.jl:21) */
    int64_t n_ext;      const double* ext;       /* parameter blocks of the aspheric primitives (see bmo_prim_type)       */
    int32_t n_jones;    const double* jones;     /* [n_jones][10]: GlobalJonesBasis of a PolarizationFilter, 3x3 real row-major
                                                    (XZBasis(1,0,0,0) by default), then its cutoff (PolarizationFilter.jl:5-9) */
    int32_t norm_zero_rule;                      /* 1 (use this): zero-vector norm of duals is a clean zero -- pinned by test/runtests.jl:1309-1314; 0: NaN partials */
    int32_t reserved;
} bmo_tables;

typedef struct bmo_ctx bmo_ctx;        /* one per process and GPU                                  */
typedef struct bmo_sys bmo_sys;        /* device copy of a flattened System                        */
typedef struct bmo_result bmo_result;  /* device-resident result of one trace call                 */

/* flags of bmo_trace_* */
#define BMO_KEEP_SEGMENTS 1u  /* keep the full segment table (needed to rebuild Beam trees / run the PD kernel) */
#define BMO_INPUT_DEVICE 2u   /* input arrays are device pointers (already resident in HBM)        */
/* flag of bmo_pd_accumulate*: evaluate every pixel-beamlet pair in the reference's operation order
 * (slower; the default kernel is algebraically identical, strength-reduced, within 1e-8 rel. L2)   */
#define BMO_PD_REFERENCE_ORDER 4u
/* flag of bmo_trace_rays / bmo_trace_rays_spots: `dir` holds ONE direction [3] shared by every ray of the bundle (a
 * collimated source, BeamGroups.jl:51-120 / :232-243: every beam of the group is built with the same `dir`), so a
 * host bundle ships 24 B per ray instead of 48.  lambda_id == NULL already means "all rays use lambdas[0]".     */
#define BMO_UNIFORM_DIR 8u

typedef struct bmo_counters {
    int64_t interactions;   /* hits that reached interact3d (a Gaussian triple counts 3)           */
    int64_t sdf_evals;      /* primitive-SDF evaluations (value or dual)                           */
    int64_t tri_tests;      /* Moeller-Trumbore evaluations                                        */
    int64_t waves;          /* wavefront iterations (bounces)                                      */
    int64_t kernel_launches;/* CUDA kernels launched by the library since the last reset           */
    int64_t px_beamlets;    /* pixel-beamlet pairs accumulated by bmo_pd_accumulate                */
    double trace_ms;        /* device time of the last trace call (CUDA events on the ctx stream)  */
    double pd_ms;           /* device time of the last bmo_pd_accumulate                           */
    double trace_step_ms;   /* accumulated device time of the trace_step kernel (K1) since the reset  */
    int64_t trace_step_launches;
    double scatter_ms;      /* accumulated device time of the queue scatter kernel (K3)             */
    double scatter_bytes;   /* algorithmic bytes moved by K3 (read + write of the surviving rays)   */
    double pd_field_ms;     /* accumulated device time of the pd_field kernel (K4)                  */
    int64_t psf_pairs;      /* pixel-hit pairs summed by bmo_psf_intensity                          */
    double psf_ms;          /* device time of the last psf_intensity kernel (K6)                    */
} bmo_counters;

int32_t bmo_init(int32_t device, bmo_ctx** ctx);
int32_t bmo_shutdown(bmo_ctx* ctx);   /* free the systems, results and sources made on ctx first: their free calls use the context */
const char* bmo_last_error(void);
int32_t bmo_set_stream(bmo_ctx* ctx, void* cuda_stream);  /* cudaStream_t; NULL = legacy default  */
int32_t bmo_counters_get(bmo_ctx* ctx, bmo_counters* out);
int32_t bmo_counters_reset(bmo_ctx* ctx);

/* replaces: construction of System / StaticSystem + Leaves flattening (System.jl:10-45)          */
int32_t bmo_system_upload(bmo_ctx* ctx, const bmo_tables* tables, bmo_sys** sys);
int32_t bmo_system_free(bmo_sys* sys);
/* Batched kinematic poses (replaces translate3d!/rotate3d! between solves, AbstractShape.jl:56-94,
 * Mesh.jl:78-96): pose p uses prims[p*n_prims ...], vertices[p*n_vertices ...], bounds[p*n_parts*10 ...].
 * Rays select their pose with pose_id.  n_poses = 1 restores the uploaded tables.                */
int32_t bmo_system_set_poses(bmo_sys* sys, int32_t n_poses, const bmo_prim* prims, const double* vertices,
                             const double* bounds, const double* det_pos /* [n_poses][n_objects][3] */,
                             const double* det_dir /* [n_poses][n_objects][9] */);

/* ---- K5: batched kinematics on the device ----------------------------------------------------------------
 * replaces: the loop `translate3d!(obj, ...) / rotate3d!(obj, axis, theta)` over many poses of one system
 * (AbstractShape.jl:56-94, AbstractShapeTrait.jl:88-128, UnionSDF.jl:63-82, Mesh.jl:78-96, ObjectGroups.jl:21-47,
 * rotate3d LinearAlgebraUtils.jl:55-65; pose sweeps: test/runtests.jl:2092-2120) followed by re-flattening.
 * The flattener uploads the kinematic tree of the system once (bmo_system_set_kinematics); a sweep is a short program of
 * micro-ops, the same for every pose, whose numeric operands (offset vectors, rotation matrices) vary per pose.  One CUDA
 * block per pose replays the program on the tree with the reference's operation order (`pos + offset`, `R * dir`, pivot
 * rule `v = (R * v) - v`, mesh `(V - p) * R' + p`, no FMA contraction) and writes that pose's prim records, vertices,
 * detector poses and part bounds -- the tables bmo_system_set_poses would have been handed.
 * Nodes are laid out in pre-order, so a subtree is the index range [i, i + size).                                   */
enum bmo_kin_kind {
    BMO_KIN_GROUP = 0,   /* ObjectGroup: own center + dir (ObjectGroups.jl:21-35)                                       */
    BMO_KIN_MULTI = 1,   /* MultiShape object: no own pose; position = position of its pivot child (AbstractShapeTrait.jl:77-84;
                            PlateBeamsplitter: the coating)                                                          */
    BMO_KIN_UNION = 2,   /* UnionSDF: own pos + dir, members keep world poses (UnionSDF.jl:63-82)                     */
    BMO_KIN_PRIM = 3,    /* one prim record (a primitive, or a meniscus frame whose children are posed relative to it) */
    BMO_KIN_MESH = 4     /* Mesh: pos, dir and world-space vertices (Mesh.jl:78-96)                                   */
};
typedef struct bmo_kin_node {
    int32_t kind;
    int32_t size;      /* nodes of the subtree rooted here, this one included                                          */
    int32_t pos_ref;   /* node whose stored position is position(node): itself, or (MULTI) the pivot child's pos_ref    */
    int32_t index;     /* PRIM: prim record; MESH: mesh index; else -1                                                 */
    int32_t flags;     /* bit 0: SphereSDF -- orientation!(::SphereSDF) is a no-op (SphericalLensSDF.jl:82-84)          */
    int32_t object;    /* object whose detector pose (bmo_object.pos / .dir) follows this node, else -1               */
    double pos[3];     /* position(node) at upload                                                                    */
    double dir[9];     /* orientation(node) at upload, row-major                                                      */
} bmo_kin_node;
enum bmo_kin_op_kind {
    BMO_KIN_TRANSLATE = 0,     /* every node of subtree(node): pos = pos + param[0..2]; mesh vertices likewise          */
    BMO_KIN_TRANSLATE_TO = 1,  /* offset = param[0..2] - position(node), then as TRANSLATE (translate_to3d!)            */
    BMO_KIN_ROT_FRAME = 2,     /* dir(node) = R * dir(node), R = param[0..8] row-major (GROUP, UNION)                    */
    BMO_KIN_ROT_LEAF = 3,      /* PRIM: dir = R * dir (unless SphereSDF); MESH: V = (V - pos) * R' + pos, dir = R * dir   */
    BMO_KIN_PIVOT = 4          /* v = position(node) - position(pivot); v = (R * v) - v; TRANSLATE subtree(node) by v    */
};
typedef struct bmo_kin_op { int32_t kind, node, pivot, param; } bmo_kin_op;
/* prim_bounds: [n_prims][10] = bounding sphere (centre xyz, radius) and box (lo xyz, hi xyz) of every top-level prim record
 * in its own frame (meniscus: in the frame of the meniscus record; entries of meniscus children are ignored).          */
int32_t bmo_system_set_kinematics(bmo_sys* sys, int32_t n_nodes, const bmo_kin_node* nodes, const double* prim_bounds);
/* params: [n_poses][n_params][9] doubles.  Starts from the uploaded tables (pose 0 of bmo_system_upload) for every pose;
 * afterwards the system holds n_poses poses exactly as after bmo_system_set_poses.                                   */
int32_t bmo_system_apply_poses(bmo_sys* sys, int32_t n_poses, int32_t n_ops, const bmo_kin_op* ops, int32_t n_params, const double* params);
/* read back the tables of one pose (tests / debugging): any pointer may be NULL.  prims: [n_prims] records,
 * vertices: [n_vertices][3], bounds: [n_parts][10], det_pose: [n_objects][12] (pos, dir row-major).                    */
int32_t bmo_system_get_pose(bmo_sys* sys, int32_t pose, bmo_prim* prims, double* vertices, double* bounds, double* det_pose);

/* replaces: solve_system!(system, beams(bg)) for Beam{Ray} / Beam{PolarizedRay}
 * (System.jl:130-154, 444-475).  pos/dir: [n][3]; lambda_id: [n] index into tables.lambdas;
 * E0: NULL or [n][6] (re,im x 3) -> PolarizedRay; pose_id: NULL or [n].                          */
int32_t bmo_trace_rays(bmo_sys* sys, int64_t n, const double* pos, const double* dir, const int32_t* lambda_id,
                       const double* E0, const int32_t* pose_id, int32_t r_max, uint32_t flags, bmo_result** out);

/* bmo_trace_rays + bmo_result_spots in one call, for systems without beamsplitters (one beam per ray):
 * replaces `solve_system!(system, beams(bg))` followed by reading `Spotdetector.data`
 * (System.jl:463-468, Spotdetector.jl:50-61).  det_object (NULL ok) / xz: [n] / [n][2] host arrays; xz of a ray that
 * reached no Spotdetector is (NaN, NaN), so det_object is only needed to tell several detectors apart.
 * With host inputs the rays are traced in sub-batches on separate streams, so that the host->device
 * copy of one sub-batch and the device->host copy of the hits of another overlap the waves of a
 * third (pinned host memory makes the copies truly asynchronous).  out may be NULL.              */
int32_t bmo_trace_rays_spots(bmo_sys* sys, int64_t n, const double* pos, const double* dir, const int32_t* lambda_id,
                             const double* E0, const int32_t* pose_id, int32_t r_max, uint32_t flags,
                             int32_t* det_object, double* xz, bmo_result** out);

/* replaces: solve_system!(system, ::GaussianBeamlet) (System.jl:274-318) for n root beamlets.
 * rays: [n][3 (chief, waist, divergence)][6 (pos, dir)]; w0, E0 (re,im): beamlet fields
 * (Gaussian.jl:33-42).                                                                           */
int32_t bmo_trace_beamlets(bmo_sys* sys, int64_t n, const double* rays, const int32_t* lambda_id, const double* w0,
                           const double* E0, const int32_t* pose_id, int32_t r_max, uint32_t flags, bmo_result** out);

/* replaces: solve_system!(system, beam; retrace = true) for beams that already hold a solution
 * (solve_system!, System.jl:444-461; retrace_system! for Beam, :188-255, and GaussianBeamlet, :326-428).
 * `prev` is the result of an earlier bmo_trace_* / bmo_retrace call (with its segment table) on a system
 * of the same structure; `sys` carries the poses after the kinematic changes.  Every beam of the previous
 * tree re-validates its stored path: each stored ray is intersected only with the object it hit before
 * (or with the shape hinted by the preceding interaction) and interacts again; where the path breaks the
 * stored tail and children are dropped and the ordinary non-sequential trace continues from there with no
 * hint.  Children of a re-validated beamsplitter hit keep retracing their own stored paths, and Gaussian
 * children keep their stored w0 (_modify_beam_head!, Gaussian.jl:154-162).  Like the reference, a retraced
 * ray does not see objects that moved into its path.  The roots restart from their stored first rays.    */
int32_t bmo_retrace(bmo_sys* sys, bmo_result* prev, int32_t r_max, uint32_t flags, bmo_result** out);

/* ---- result access.  Beams are numbered roots first (0..n-1), children in spawn order.         */
typedef struct bmo_result_info {
    int64_t n_roots, n_beams, n_segments /* -1 until bmo_result_beams / _segments was called on a spot-only trace */, interactions;
    int32_t rays_per_beam;  /* 1 (Beam) or 3 (GaussianBeamlet: chief, waist, divergence)          */
    int32_t polarized;
    int32_t waves;
    int32_t reserved;
} bmo_result_info;
int32_t bmo_result_get_info(bmo_result* r, bmo_result_info* info);
/* per beam: parent beam (-1 for roots), index of the child within its parent (0 transmitted, 1 reflected),
 * number of segments, status of the last segment (bmo_status), first segment row.
 * Gaussian extras (NULL ok): w0, E0 (re,im), lambda_id.                                          */
int32_t bmo_result_beams(bmo_result* r, int32_t* parent, int32_t* child_slot, int32_t* n_seg, int32_t* status,
                         int64_t* first_seg, double* w0, double* E0, int32_t* lambda_id);
/* segment table, beam-major; rows = n_segments * rays_per_beam (Gaussian: chief, waist, div interleaved).
 * Any pointer may be NULL.  t = Inf <=> intersection === nothing.  E0: [rows][6].                 */
int32_t bmo_result_segments(bmo_result* r, double* pos, double* dir, double* n, double* t, double* nrm,
                            int32_t* object, int32_t* part, double* E0);
/* Spotdetector hits (Spotdetector.jl:50-61): per beam the detector object index (-1: none) and local (x, z). */
int32_t bmo_result_spots(bmo_result* r, int32_t* det_object, double* xz);
/* same, but leaves the data on the device: returns device pointers valid until bmo_result_free   */
int32_t bmo_result_spots_device(bmo_result* r, const int32_t** det_object, const double** xz);
int32_t bmo_result_free(bmo_result* r);

/* ---- sources generated on the device (bmo_source.cu) -----------------------------------------------------
 * replaces: building the rays of UniformDiscSource (BeamGroups.jl:222-245), CollimatedSource (:152-195) and PointSource
 * (:51-100) on the host and copying them over.  The host computes every transcendental and every per-ring quantity (ring
 * counts, rotate3d matrices, the basis) with the same code that builds its own bundles; the device expands the descriptor.
 *   disc:        one thread per ray k: rho = sqrt((k + 0.5) / n), phi = k * phi0, r = radius * rho,
 *                pos = pos + ((r cos phi) e1 + (r sin phi) e2); dir = `dir` for every ray.  CUDA's double sin / cos are not
 *                correctly rounded: positions agree with the host to a few ulp, not to the bit.
 *   collimated:  ray 0 = pos; ring ray j = pos + v_j with v_0 = ring.start (= r b1), v_{j+1} = ring.rot v_j;
 *                dir = `dir` for every ray.
 *   point:       pos for every ray; ray 0 has direction `dir`; ring ray j has v_j renormalised like RayBundle
 *                (v * (1 / sqrt(vx vx + vy vy + vz vz))), v_0 = ring.start (= the ring's first direction).
 * Ring sources run one thread per ring through the serial recurrence in linalg.matvec's operation order without FMA
 * contraction, so they are bit-identical to the host constructors.                                               */
enum bmo_source_kind { BMO_SRC_DISC = 0, BMO_SRC_COLLIMATED = 1, BMO_SRC_POINT = 2 };
typedef struct bmo_source_ring {
    int64_t first, count;   /* rays [first, first + count); rings are contiguous from ray 1; count 0 = skipped ring  */
    double start[3];        /* collimated: first offset r * b1; point: first direction                                */
    double rot[9];          /* rotate3d(dir, 2 pi / count), row-major                                                 */
} bmo_source_ring;
typedef struct bmo_source_desc {
    int32_t kind;           /* bmo_source_kind                                                                        */
    int32_t reserved;
    int64_t n_rays;
    int64_t n_rings;        /* ring sources: sum of the counts = n_rays - 1; discs: 0                                */
    const bmo_source_ring* rings;   /* host array [n_rings]                                                          */
    double pos[3];
    double dir[3];          /* normalised the way RayBundle stores it                                                 */
    double e1[3], e2[3];    /* disc basis (e2 = normalize(dir x e1))                                                 */
    double radius, phi0;    /* disc: diameter / 2, 2 pi / (1 + sqrt 5)                                                 */
} bmo_source_desc;
typedef struct bmo_source bmo_source;
/* Fills the device buffers of *src from the context's pool, enqueued on the context's stream.  BMO_EINVAL for an
 * unknown kind, n_rays < 1, a non-finite value or rings that do not tile [1, n_rays).                             */
int32_t bmo_source_create(bmo_ctx* ctx, const bmo_source_desc* desc, bmo_source** src);
/* Pose-tiled source for a pose sweep: replaces building the same source once per step of the loop `translate3d!(obj, ...)
 * -> empty!(sd) -> solve_system!(system, source) -> sd.data` (AbstractShape.jl:56-94, Spotdetector.jl:50-61,
 * System.jl:444-468).  n_poses copies of the descriptor's rays, pose-major: ray i is ray i mod n_rays of the descriptor and
 * pose_id[i] = i / n_rays, so every tile is bit-identical to bmo_source_create (discs keep rho = sqrt((k + 0.5) / n_rays);
 * ring sources run their recurrence once and copy it).  bmo_source_create is the n_poses = 1 case.  BMO_EINVAL also for
 * n_poses < 1 or n_rays * n_poses overflowing int64.                                                              */
int32_t bmo_source_create_poses(bmo_ctx* ctx, const bmo_source_desc* desc, int32_t n_poses, bmo_source** src);
/* Source slice, for sharding one source over several GPUs or tracing it in pieces: rays [first, first + count) of the one-pose
 * source bmo_source_create would make, bit for bit (discs: to the same bits as those rays of the unsliced source, not closer
 * to the host than it is).  A disc computes ray first + i with rho = sqrt((k + 0.5) / n_rays); each ring that overlaps the
 * slice runs its recurrence from its own start and writes the rays inside the slice; ray 0 is written only when first == 0.
 * bmo_source_device reports n = count, bmo_source_rays copies the slice, bmo_source_pose_ids gives NULL.  BMO_EINVAL for
 * first < 0, count < 1, first + count > n_rays, and whatever bmo_source_create refuses.                              */
int32_t bmo_source_create_slice(bmo_ctx* ctx, const bmo_source_desc* desc, int64_t first, int64_t count, bmo_source** src);
/* Device pose ids [n_rays * n_poses] for bmo_trace_rays(..., pose_id, BMO_INPUT_DEVICE) or, of a beamlet source,
 * bmo_trace_beamlets; NULL for a one-pose source.  Valid until bmo_source_free.                                      */
int32_t bmo_source_pose_ids(bmo_source* src, int32_t* n_poses, const int32_t** pose_id);
/* Device pointers for bmo_trace_rays(..., BMO_INPUT_DEVICE | (*uniform_dir ? BMO_UNIFORM_DIR : 0)): pos [n][3];
 * dir [n][3], or one direction [3] when *uniform_dir is 1.  n counts the rays of every pose.  Valid until bmo_source_free.
 * BMO_EINVAL on a beamlet source (bmo_source_create_beamlets).                                                          */
int32_t bmo_source_device(bmo_source* src, int64_t* n, const double** pos, const double** dir, int32_t* uniform_dir);
/* host copies (NULL ok): pos [n][3], dir [n][3] (a uniform direction is expanded to every ray); BMO_EINVAL on a
 * beamlet source                                                                                                 */
int32_t bmo_source_rays(bmo_source* src, double* pos, double* dir);
int32_t bmo_source_free(bmo_source* src);   /* before bmo_shutdown of the source's context */

/* ---- Gaussian beamlet sources generated on the device ----------------------------------------------------------------
 * replaces: BeamletBundle.from_params / GaussianBeamlet (Gaussian.jl:215-256) over the rays of a disc or collimated source, built
 * on the host and copied over (144 B of rays, w0, E0 and a wavelength id per beamlet, once per pose for a pose sweep).  Every
 * beamlet shares one set of parameters; the host computes every scalar and vector below with the code of from_params, and the
 * device only adds and multiplies, in from_params' order, without FMA contraction.  Beamlet i at source position P (the
 * position bmo_source_rays gives ray i of the same source descriptor):
 *   chief       pos P,                 dir dv
 *   waist       pos P + s * w0,        dir dv
 *   divergence  pos P + s * div_offset, dir dd
 *   w0[i] = w0, E0[i] = E0.
 * With d = normalize(direction), s = normalize(support), tan_t = tan(M2 lambda / (pi w0)), I0 = 2 P0 / (pi w0^2):
 * dv = normalize(d), dd = normalize(normalize(d + tan_t s)), div_offset = -z0 tan_t, E0 = sqrt(2 I0 Z0) + 0i.       */
typedef struct bmo_beamlet_desc {
    double dv[3];           /* chief and waist direction                                                             */
    double dd[3];           /* divergence direction                                                                  */
    double s[3];            /* normalised support vector                                                             */
    double w0;              /* waist radius, > 0                                                                     */
    double div_offset;      /* -z0 tan_t: offset of the divergence ray along s                                      */
    double E0[2];           /* field amplitude (re, im)                                                              */
} bmo_beamlet_desc;
/* Beamlets [first, first + count) of the one-pose source, tiled n_poses times pose-major (beamlet i is beamlet first + i mod
 * count, pose_id[i] = i / count; n_poses > 1 only for the whole source, first = 0 and count = n_rays).  The positions are those
 * bmo_source_create_slice / _poses give the same descriptor, so each tile and slice has the bits of the matching rows of the
 * whole one-pose source.  BMO_EINVAL for whatever bmo_source_create refuses, a point source (its directions differ per ray),
 * non-finite constants, w0 <= 0, n_poses < 1, n_poses > 1 on a slice, a slice outside the source and count * n_poses
 * overflowing int64.  bmo_source_device and bmo_source_rays refuse a beamlet source with BMO_EINVAL; bmo_source_pose_ids
 * gives its pose ids (NULL for one pose).                                                                                */
int32_t bmo_source_create_beamlets(bmo_ctx* ctx, const bmo_source_desc* desc, const bmo_beamlet_desc* beamlet, int32_t n_poses,
                                   int64_t first, int64_t count, bmo_source** src);
/* Device pointers for bmo_trace_beamlets(..., BMO_INPUT_DEVICE) (lambda_id NULL: the source's one wavelength is lambdas[0]):
 * rays [n][3][6], w0 [n], E0 [n][2]; n counts the beamlets of every pose.  Valid until bmo_source_free.  BMO_EINVAL on a ray
 * source.                                                                                                                 */
int32_t bmo_source_beamlets_device(bmo_source* src, int64_t* n, const double** rays, const double** w0, const double** E0);
/* host copies (NULL ok): rays [n][3][6], w0 [n], E0 [n][2].  BMO_EINVAL on a ray source.                                  */
int32_t bmo_source_beamlets(bmo_source* src, double* rays, double* w0, double* E0);

/* ---- spot-diagram reduction on the device --------------------------------------------------------------
 * replaces: reading Spotdetector.data (Spotdetector.jl:50-61) back to compute what a spot diagram shows.  Works over the
 * n_beams * R entries bmo_result_spots reports with det_object[k] == det_object (a beamlet result counts chief, waist and
 * divergence).  rms = sqrt(sum((x - cx)^2 + (z - cz)^2) / hits) in a second pass; max_r = max sqrt(x x + z z) about the
 * detector origin; with no hits every floating field is NaN.  The sums run over a fixed partition of the entry index
 * whose partials are combined in index order, so two calls give the same bits; hits, outside, max_r, lo / hi and the
 * histogram are exact.  The partition (part of this contract: bmo_spot_stats_results and bmo_spot_stats_sharded use it on
 * the total of their entries, and the sharded call needs shards cut to it) gives each block BMO_SPOT_PER(m) consecutive
 * entries of the m entries reduced, the last block the rest.
 * window (NULL ok, required with counts): x_lo, x_hi, z_lo, z_hi, finite with hi > lo; a hit outside the closed window
 * counts in `outside`.  counts (NULL ok): [nz][nx], counts[j * nx + i] = hits with
 * i = min(floor((x - x_lo) / (x_hi - x_lo) * nx), nx - 1), j likewise in z; overwritten.  Host pointer, or device
 * pointer with BMO_INPUT_DEVICE.  (The struct cannot share the function's name in C, hence bmo_spot_info.)        */
/* entries per block of the partition of m spot entries: 4096 * max(1, ceil(m / (4096 * 1024))), so <= 1024 blocks          */
#define BMO_SPOT_PER(m) (4096 * (((m) + 4096 * 1024 - 1) / (4096 * 1024) > 1 ? ((m) + 4096 * 1024 - 1) / (4096 * 1024) : 1))
typedef struct bmo_spot_info {
    int64_t hits;
    int64_t outside;
    double centroid[2];     /* mean x, mean z          */
    double rms;
    double max_r;
    double lo[2], hi[2];    /* min / max of x and z    */
} bmo_spot_info;
int32_t bmo_spot_stats(bmo_result* r, int32_t det_object, const double* window, int32_t nx, int32_t nz, bmo_spot_info* out,
                       int64_t* counts, uint32_t flags);
/* Per-pose spot statistics of a pose sweep: replaces reading sd.data after every step of the loop `translate3d!(obj, ...)
 * -> empty!(sd) -> solve_system!(system, source) -> sd.data` (AbstractShape.jl:56-94, Spotdetector.jl:50-61,
 * System.jl:444-468).  out[p] is bmo_spot_stats's definition over the entries of the beams whose pose is p (all R entries
 * of a beamlet; children inherit their root's pose), taken in increasing entry index; counts (NULL ok): [n_poses][nz][nx]
 * over the shared window, host pointer, or device pointer with BMO_INPUT_DEVICE.  The beams are ordered stably by pose and
 * each pose's entries are cut into slices by bmo_spot_stats's formula on that pose's entry count, so out[p] has the bits
 * bmo_spot_stats gives for a one-pose result that lists the pose's entries in the same order (always the case without
 * beamsplitters: the roots follow the input order).  n_poses must be the pose count of the system at trace time
 * (BMO_EINVAL otherwise), and bmo_spot_stats's argument checks apply.                                               */
int32_t bmo_spot_stats_poses(bmo_result* r, int32_t det_object, int32_t n_poses, const double* window, int32_t nx, int32_t nz,
                             bmo_spot_info* out, int64_t* counts, uint32_t flags);
/* Spot statistics over several results on one device: replaces reading sd.data after several solve_system! calls into one
 * Spotdetector without empty!(sd) in between (Spotdetector.jl:50-61): field points, one source per wavelength, or a bundle
 * traced in pieces.  bmo_spot_stats's definition over the concatenation of the results' entries, the results in list order and
 * each result's entries in entry order; the partition is BMO_SPOT_PER of the total entry count N = sum n_beams * R, and a
 * block may straddle two results.  The output has the bits of bmo_spot_stats on one result that lists the same entries in the
 * same order: without beamsplitters a bundle traced as k slices gives the bits of tracing it once, however it is cut.  The
 * results must share one context and det_object must be a Spotdetector of every result's system; R = 1 and R = 3 results
 * mix; poses are ignored.  BMO_EINVAL for n_results < 1, a NULL entry, and whatever bmo_spot_stats refuses.            */
int32_t bmo_spot_stats_results(int32_t n_results, bmo_result* const* results, int32_t det_object, const double* window,
                               int32_t nx, int32_t nz, bmo_spot_info* out, int64_t* counts, uint32_t flags);

enum bmo_status {
    BMO_ST_ACTIVE = 0,
    BMO_ST_MISS = 1,      /* no intersection: beam leaves the system                               */
    BMO_ST_ABSORBED = 2,  /* interact3d returned nothing (detector, stop, unsupported pairing)     */
    BMO_ST_RMAX = 3,      /* r_max segments reached (System.jl:133)                                */
    BMO_ST_SPLIT = 4,     /* beamsplitter: children spawned, parent stops                          */
    BMO_ST_CLIPPED = 5,   /* Gaussian: waist or divergence ray missed (System.jl:288-296)          */
    BMO_ST_TORN = 6,      /* Gaussian: rays hit different shapes (System.jl:298-304)               */
    BMO_ST_ERROR = 7      /* reference would throw ArgumentError (non-unit dir / normal in refraction3d) */
    /* status & 0x100: a PolarizedRay's E0 failed the reference's orthogonality check (|dir.E0| <= 1e-14,
       PolarizedRays.jl:54-56) somewhere along the beam; the reference throws, the tracer flags and continues */
};

/* replaces: interact3d(::AbstractSystem, ::Photodetector, ::GaussianBeamlet, ray_id)
 * (Photodetector.jl:69-107) summed over every leaf beamlet of `r` whose chief ray ends on detector
 * `pd_object`, for pose `pose`.  field: n*n complex128, column-major [i, j] (re,im interleaved),
 * host pointer, or device pointer if flags has BMO_INPUT_DEVICE; the result is ADDED to it (the
 * reference's `+=`).                                                                             */
int32_t bmo_pd_accumulate(bmo_sys* sys, bmo_result* r, int32_t pd_object, int32_t pose, double* field, uint32_t flags);
/* batched form for pose sweeps: fields[pose] for pose in [0, n_poses)                             */
int32_t bmo_pd_accumulate_poses(bmo_sys* sys, bmo_result* r, int32_t pd_object, int32_t n_poses, double* fields, uint32_t flags);
/* optical_power(pd) = trapz((x, y), |E|^2 / (2 Z0)) (Photodetector.jl:109-116) on the device.    */
int32_t bmo_pd_power(bmo_sys* sys, int32_t pd_object, int32_t n_fields, const double* fields, double* power, uint32_t flags);

/* ---- PSFDetector (OpticalComponents/Detectors/PSFDetector.jl) ---------------------------------------
 * bmo_psf is the detector's `data::Vector{PSFData}` on the device.
 * bmo_psf_collect replaces interact3d(::AbstractSystem, ::PSFDetector, ::Beam{T, Ray{T}}, ::Ray) (:77-89) for every
 * beam of `r` that ended on `psf_object`: hit position, direction, optical_path_length(beam) (through the
 * parents), |dir . normal| and 2 pi / lambda are appended to *psf (created when *psf == NULL; the reference's
 * detector also accumulates until empty!).  `r` must hold its segment table; PolarizedRay results add nothing
 * (no interact3d method, AbstractSystem.jl:30-33).
 * GaussianBeamlet results (Gaussian.jl:124-135): every beamlet absorbed with its chief ray on `psf_object` appends three
 * records, chief, waist, divergence, each from its own ray's last hit (position, direction, |dir . normal|) with the
 * beamlet's 2 pi / lambda.  OPL: the chief's is the OPL of the parent's chief beam (the children of a beamsplitter link only
 * their chief beam to the parent, Gaussian.jl:107-111), at any depth of the beamlet tree, plus the chief's own t * n in
 * order; the waist's and divergence's are their own t * n only.  A torn or clipped beamlet appends nothing.         */
typedef struct bmo_psf bmo_psf;
int32_t bmo_psf_collect(bmo_sys* sys, bmo_result* r, int32_t psf_object, bmo_psf** psf, int64_t* n_total);
int32_t bmo_psf_count(bmo_psf* psf, int64_t* n);
/* host copy of the records: [n][9] = hit xyz, dir xyz, opl, proj, k (PSFData, :1-7)                         */
int32_t bmo_psf_data(bmo_psf* psf, double* records);
/* calc_local_lims(psf; crop_factor, center) (:112-141): center 0 = :centroid, 1 = :bbox; lims = x_min, x_max, z_min, z_max */
int32_t bmo_psf_lims(bmo_sys* sys, bmo_psf* psf, int32_t psf_object, int32_t pose, double crop_factor, int32_t center, double* lims);
/* intensity(psf; n, ...) (:190-237) on xs = LinRange(lims[0], lims[1], n) .+ x0_shift, zs likewise:
 * intensity[i + n*j] = |sum_h proj_h cis(k_h (opl_h + (p_ij - hit_h) . dir_h))|^2 (raw, unscaled).  Host pointer, or
 * device pointer with BMO_INPUT_DEVICE.                                                                     */
int32_t bmo_psf_intensity(bmo_sys* sys, bmo_psf* psf, int32_t psf_object, int32_t pose, int32_t n, const double* lims,
                          double x0_shift, double z0_shift, double* intensity, uint32_t flags);
/* Columns [j0, j1) of bmo_psf_intensity's map: intensity[i + n*(j - j0)] for j in [j0, j1), n * (j1 - j0) doubles, with the bits
 * bmo_psf_intensity gives those pixels (a pixel's sum depends only on (i, j), lims, the shifts and the records in order).  Host
 * pointer, or device pointer with BMO_INPUT_DEVICE.  BMO_EINVAL unless 0 <= j0 <= j1 <= n (an empty range writes nothing); otherwise
 * bmo_psf_intensity's checks.  The building block of a column-sharded map for a host that brings its own transport.           */
int32_t bmo_psf_intensity_cols(bmo_sys* sys, bmo_psf* psf, int32_t psf_object, int32_t pose, int32_t n, const double* lims,
                               double x0_shift, double z0_shift, int32_t j0, int32_t j1, double* intensity, uint32_t flags);
int32_t bmo_psf_free(bmo_psf* psf);   /* empty!(psf) */

/* pose sweep in one call: replaces the loop `translate3d!(mirror, ...); empty!(pd); solve_system!(system, beam);
 * optical_power(pd)` (test/runtests.jl:2092-2120, docs/src/tutorials/michelson.md:251-256) after the batched trace:
 * fields[pose] start from zero on the device, power[pose] = optical_power of each; fields (host, [n_poses][n*n*2]) and
 * power (host, [n_poses]) may each be NULL -- with fields == NULL only n_poses doubles leave the device.        */
int32_t bmo_pd_sweep(bmo_sys* sys, bmo_result* r, int32_t pd_object, int32_t n_poses, double* fields, double* power, uint32_t flags);

/* ---- multi-GPU: the one exchange step of the path ---------------------------------------------------------
 * replaces: the serial `for beam in beams(bg)` of solve_system!(system, ::AbstractBeamGroup) (System.jl:463-468) once the
 * host shards the beams of a group over several GPUs -- every GPU accumulates its beamlets onto a full n x n partial field
 * (bmo_pd_accumulate) and the partial fields are summed, which is what the reference's `pd.field[i, j] += ...`
 * (Photodetector.jl:103) does serially.  One complex128 all-reduce over NVLink (NCCL, bound at run time: dlopen of
 * libnccl.so.2, or BMO_NCCL_LIB).  Tracing itself needs no communication (rays / beamlets are independent).
 *   one process per GPU: rank 0 calls bmo_comm_unique_id, ships the 128 bytes to the other ranks, all call bmo_comm_init;
 *   one process, n GPUs: bmo_comm_init_local over the n contexts + bmo_pd_allreduce_local (grouped).                  */
#define BMO_COMM_ID_BYTES 128
#define BMO_COMM_SYNC 16u   /* flag: synchronise the context's stream before returning (device fields; host fields always do) */
typedef struct bmo_comm bmo_comm;
int32_t bmo_comm_unique_id(uint8_t* id /* [BMO_COMM_ID_BYTES] */);
int32_t bmo_comm_init(bmo_ctx* ctx, int32_t n_ranks, int32_t rank, const uint8_t* id, bmo_comm** comm);
int32_t bmo_comm_init_local(int32_t n, bmo_ctx* const* ctxs, bmo_comm** comms /* [n] out */);
int32_t bmo_comm_info(bmo_comm* comm, int32_t* rank, int32_t* n_ranks, int32_t* nccl_version);
/* field: n_complex complex128 values (re, im interleaved; a Photodetector field has n_complex = n * n), summed in place over
 * all ranks.  Host pointer (staged through the device), or device pointer with BMO_INPUT_DEVICE (enqueued on the context's
 * stream; add BMO_COMM_SYNC to wait for it).                                                                    */
int32_t bmo_pd_allreduce(bmo_comm* comm, double* field, int64_t n_complex, uint32_t flags);
int32_t bmo_pd_allreduce_local(int32_t n, bmo_comm* const* comms, double* const* fields, int64_t n_complex, uint32_t flags);
/* Spot statistics of a ray bundle sharded over ranks, collective: every rank of comm passes the result of its shard (NULL
 * on a rank whose shard holds no rays); every rank receives the statistics (and histogram) of the concatenation of all
 * ranks' entries in rank order, with the bits bmo_spot_stats_results gives for the shard results in rank order -- for
 * aligned, splitter-free shards of one source the bits of one unsharded trace; with one rank, bmo_spot_stats's bits.
 * Every rank except the last must hold a multiple of BMO_SPOT_PER(N) entries, N the total over all ranks, so that no
 * block of the partition crosses a rank boundary.  det_object, nx, nz and the window must be the same on every rank.
 * Steps, on the context's stream: (1) all-gather of each rank's entry count, argument verdict, det_object, histogram shape
 * and window; a refusal on any rank (bmo_spot_stats's checks, another context, unaligned shards, a detector, histogram shape
 * or window that differs from rank 0's) makes every rank return the same BMO_E* code; (2) each rank reduces its entries to
 * per-block partials; (3) the partials are all-gathered and combined in global block order on every rank; (4) the same
 * for the squared distances to the centroid; (5) one int64 all-reduce (sum) of the histogram.  Only the statistics and
 * the histogram leave the device.  counts: host pointer, or device pointer with BMO_INPUT_DEVICE.  Only arguments are
 * agreed on: a CUDA or NCCL failure on one rank (an allocation, a launch) returns BMO_ECUDA / BMO_ENCCL on that rank alone
 * and leaves the other ranks waiting in the next collective, as any failed NCCL collective does.                     */
int32_t bmo_spot_stats_sharded(bmo_comm* comm, bmo_result* r, int32_t det_object, const double* window, int32_t nx, int32_t nz,
                               bmo_spot_info* out, int64_t* counts, uint32_t flags);
/* PSFDetector records of a ray bundle sharded over ranks, collective: every rank receives in *all a new handle, freed with
 * bmo_psf_free, holding all ranks' records in rank order; `local` may be NULL on a rank without hits.  Steps, on the context's
 * stream: (1) all-gather of each rank's record count and argument verdict (`local` on another context than comm, all NULL, a
 * total that overflows int64); a refusal on any rank makes every rank return the same code; (2) one all-gather of both record
 * arrays, padded to the largest count, each rank's part then copied into place.  With one rank, a device copy of `local`.  A
 * CUDA or NCCL failure returns on the failing rank alone, as in bmo_spot_stats_sharded.                                  */
int32_t bmo_psf_allgather(bmo_comm* comm, bmo_psf* local, bmo_psf** all);
/* bmo_psf_intensity over ranks, collective: every rank passes the same gathered records (bmo_psf_allgather) and arguments and
 * receives the whole n x n map (host pointer, or device pointer with BMO_INPUT_DEVICE).  Rank r sums every record into its band of
 * pixel columns [r B, min(n, (r + 1) B)), B = ceil(n / n_ranks), and the bands are all-gathered: the map has bmo_psf_intensity's
 * bits for the same records.  Step (1) all-gathers each rank's verdict (bmo_psf_intensity's checks; sys or psf on another
 * context), n, pose, psf_object, the bits of lims and of the shifts, and the record count; a refusal or a mismatch with rank 0
 * (a rank that passes its own, ungathered records holds another count) makes every rank return the same code.  With one rank
 * there is no NCCL call.  Only arguments are agreed on, as in bmo_spot_stats_sharded.                                     */
int32_t bmo_psf_intensity_sharded(bmo_comm* comm, bmo_sys* sys, bmo_psf* all, int32_t psf_object, int32_t pose, int32_t n,
                                  const double* lims, double x0_shift, double z0_shift, double* intensity, uint32_t flags);
/* bmo_pd_sweep over ranks by pose range, collective: rank k sweeps poses [first_k, first_k + count_k) of an n_poses-pose sweep.
 * Its `sys` holds those count_k poses as its poses 0 .. count_k - 1 and `r` is their trace (pose ids 0 .. count_k - 1); a rank
 * with count == 0 passes r = NULL and still takes part.  fields: this rank's [count][n*n*2] (NULL ok), never exchanged; power:
 * [n_poses] on every rank.  Both host pointers, or device pointers with BMO_INPUT_DEVICE.  Steps, on the context's stream:
 * (1) all-gather of each rank's verdict (bmo_pd_sweep's checks on its poses; sys or r on another context than comm), pd_object,
 * the detector's n, n_poses, first and count; a refusal, another pd_object, n or n_poses than rank 0's, or ranges that do not
 * tile [0, n_poses) in rank order make every rank return the same code; (2) the rank's fields and powers with bmo_pd_sweep's
 * code; (3) one all-gather of the powers, padded to the largest count, each rank's part then copied into pose order.  A pose's
 * field and power have the bits bmo_pd_sweep gives it in one sweep of all poses when the rank's trace holds the same records
 * for it in the same order (DESIGN §14).  With one rank there is no NCCL call.  Only arguments are agreed on, as in
 * bmo_spot_stats_sharded.                                                                                                     */
int32_t bmo_pd_sweep_sharded(bmo_comm* comm, bmo_sys* sys, bmo_result* r, int32_t pd_object, int32_t n_poses, int32_t first, int32_t count,
                             double* fields, double* power, uint32_t flags);
/* bmo_spot_stats_poses over ranks by pose range, collective: rank k passes the trace `r` of poses [first_k, first_k + count_k) of an
 * n_poses-pose sweep, traced through a system that holds them as its poses 0 .. count_k - 1; a rank with count == 0 passes
 * r = NULL and still takes part.  out: [n_poses] host array, counts (NULL ok): [n_poses][nz][nx] over the window, host pointer
 * or device pointer with BMO_INPUT_DEVICE; every rank receives all n_poses statistics and histograms.  Steps, on the context's
 * stream: (1) all-gather of each rank's verdict (bmo_spot_stats_poses' checks on its poses, with count as the result's pose
 * count; r on another context than comm), det_object, n_poses, histogram shape and window bits, first and count; a refusal,
 * another det_object, n_poses, histogram shape or window than rank 0's, or ranges that do not tile [0, n_poses) in rank order
 * make every rank return the same code; (2) the rank's statistics with bmo_spot_stats_poses' code; (3) one all-gather of the
 * statistics and one of the histograms, padded to the largest count, each rank's part then copied into pose order.  Each pose is
 * reduced from its own entries only, so out[p] has the bits bmo_spot_stats_poses gives pose p in one sweep of all poses when the
 * rank's trace lists the pose's entries in the same order (DESIGN §15).  With one rank there is no NCCL call.  Only arguments
 * are agreed on, as in bmo_spot_stats_sharded.                                                                                */
int32_t bmo_spot_stats_poses_sharded(bmo_comm* comm, bmo_result* r, int32_t det_object, int32_t n_poses, int32_t first, int32_t count,
                                     const double* window, int32_t nx, int32_t nz, bmo_spot_info* out /* [n_poses] */,
                                     int64_t* counts /* [n_poses][nz][nx], NULL ok */, uint32_t flags);
int32_t bmo_comm_free(bmo_comm* comm);

/* Give device memory back: the library keeps released blocks of 64 MiB and more in a per-device free list and smaller ones in
 * CUDA's stream-ordered pool, so that the next solve of the same shape allocates nothing (INTEGRATION.md, "Device memory").  A host
 * that shares the GPU with other allocators (CUDA.jl, PyTorch) calls this after a large one-off trace; bmo_shutdown does it too.
 * The reference has no counterpart (Julia's GC owns its arrays).  Returns the bytes released from the free list in *released
 * (NULL ok).                                                                                                                    */
int32_t bmo_trim(bmo_ctx* ctx, int64_t* released);

/* FP64 DFMA micro-benchmark used as the roofline denominator of the FP64-bound kernels.          */
int32_t bmo_measure_fp64_peak(bmo_ctx* ctx, double* tflops);

/* Self-check (tests): normal3d(shape, point) (AbstractSDF.jl:79-95) of the primitive record prim_idx[i] at points[i] ([n][3], world
 * coordinates), once through the written-out gradients the tracer uses for unrotated lens primitives and once through the generic
 * dual-number evaluation (ForwardDiff's rules).  out_fast / out_generic: [n][3]; they must agree bit for bit.                    */
int32_t bmo_debug_normals(bmo_sys* sys, int64_t n, const double* points, const int32_t* prim_idx, double* out_fast, double* out_generic);

#ifdef __cplusplus
}
#endif
#endif /* BMO_H */
