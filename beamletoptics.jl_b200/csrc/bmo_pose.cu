// bmo_pose.cu -- K5: batched kinematics on the device (compiled -fmad=false: the poses are bit-identical to the ones the
// reference's kinematic API produces one at a time on the host).
//
// Reference semantics replayed per pose (citations relative to /root/reference/src):
//   translate3d!(shape, offset)        pos = pos + offset                                   AbstractTypes/AbstractShape.jl:56-59
//   rotate3d!(shape, axis, theta)      dir = R * dir                                        AbstractShape.jl:78-82
//   orientation!(::AbstractSDF, dir)   transposed_dir = transpose(dir)                      SDFs/AbstractSDF.jl:20-23
//   rotate3d!(::MultiShape / ::UnionSDF / ObjectGroup)  every child rotates, then moves by v = (R * v) - v with
//                                      v = position(child) - position(parent)               AbstractShapeTrait.jl:115-128, UnionSDF.jl:69-82
//   translate3d!(mesh, offset)         vertices .+ offset'                                  Mesh.jl:78-82
//   rotate3d!(mesh, axis, theta)       (vertices .- pos') * R' .+ pos', dir = R * dir        Mesh.jl:89-96
// The rotation matrices themselves (rotate3d, Utils/LinearAlgebraUtils.jl:55-65) are formed on the host -- cos / sin of the
// host's libm, so that the device result does not depend on CUDA's last-bit rounding of the trigonometric functions -- and
// arrive as per-pose parameters.  Matrix products sum left to right like the reference's StaticArrays expressions.
#include "bmo_host.cuh"

using namespace bmo;

namespace bmo {

struct PoseParams {
    const bmo_kin_node* nodes; int32_t n_nodes;
    const bmo_kin_op* ops; int32_t n_ops;
    const double* params; int32_t n_params;       // [n_poses][n_params][9]
    const bmo_prim* prims0; int32_t n_prims;      // uploaded records (flags patched)
    const bmo_part* parts; int32_t n_parts;
    const MeshView* meshes; int32_t n_meshes;
    const double* vertices0; int64_t n_vertices;
    const double* detpose0; int32_t n_objects;    // [n_objects][12]
    const double* prim_bounds;                    // [n_prims][10]
    bmo_prim* prims; double* vertices; double* bounds; double* detpose;   // outputs, stacked per pose
    double bound_rel, bound_abs;
};

BMO_D void mat3_mul(const double* A, const double* B, double* C) {   // C = A * B, row-major, left-to-right sums
#pragma unroll
    for (int i = 0; i < 3; i++)
#pragma unroll
        for (int j = 0; j < 3; j++) C[3 * i + j] = A[3 * i] * B[j] + A[3 * i + 1] * B[3 + j] + A[3 * i + 2] * B[6 + j];
}
BMO_D V3 mat3_vec(const double* A, V3 v) {
    return mk3(A[0] * v.x + A[1] * v.y + A[2] * v.z, A[3] * v.x + A[4] * v.y + A[5] * v.z, A[6] * v.x + A[7] * v.y + A[8] * v.z);
}
BMO_D double rf32(double x) { return (double)(float)x; }

constexpr int PBLOCK = 128;

// one block per pose
__global__ void __launch_bounds__(PBLOCK) apply_poses_kernel(const PoseParams P) {
    extern __shared__ __align__(16) double s_node[];   // [n_nodes][12]: pos(3) dir(9)
    __shared__ double s_red[PBLOCK / 32][7];
    const int pose = blockIdx.x, tid = threadIdx.x;
    const double* par = P.params + (size_t)pose * P.n_params * 9;
    double* verts = P.vertices + (size_t)pose * 3 * P.n_vertices;
    for (int k = tid; k < P.n_nodes * 12; k += PBLOCK) {
        const bmo_kin_node& nd = P.nodes[k / 12];
        const int f = k % 12;
        s_node[k] = f < 3 ? nd.pos[f] : nd.dir[f - 3];
    }
    for (int64_t k = tid; k < 3 * P.n_vertices; k += PBLOCK) verts[k] = P.vertices0[k];
    __syncthreads();

    for (int o = 0; o < P.n_ops; o++) {
        const bmo_kin_op op = P.ops[o];
        const double* q = par + 9 * op.param;
        const bmo_kin_node& nd = P.nodes[op.node];
        if (op.kind == BMO_KIN_ROT_FRAME || (op.kind == BMO_KIN_ROT_LEAF && nd.kind == BMO_KIN_PRIM)) {
            if (tid == 0 && !(op.kind == BMO_KIN_ROT_LEAF && (nd.flags & 1))) {
                double* d = s_node + 12 * op.node + 3;
                double old[9], nw[9];
                for (int k = 0; k < 9; k++) old[k] = d[k];
                mat3_mul(q, old, nw);
                for (int k = 0; k < 9; k++) d[k] = nw[k];
            }
            __syncthreads();
            continue;
        }
        if (op.kind == BMO_KIN_ROT_LEAF) {   // MESH
            const MeshView mv = P.meshes[nd.index];
            const V3 p = mk3(s_node[12 * op.node], s_node[12 * op.node + 1], s_node[12 * op.node + 2]);
            for (int64_t i = tid; i < mv.n_vertices; i += PBLOCK) {
                double* v = verts + 3 * (mv.first_vertex + i);
                V3 d = mk3(v[0] - p.x, v[1] - p.y, v[2] - p.z);
                if (mv.f32) d = mk3(rf32(d.x), rf32(d.y), rf32(d.z));
                const V3 r = mat3_vec(q, d);          // row i of (d' * R') = R[i,:] . d
                V3 w = mk3(r.x + p.x, r.y + p.y, r.z + p.z);
                if (mv.f32) w = mk3(rf32(w.x), rf32(w.y), rf32(w.z));
                v[0] = w.x; v[1] = w.y; v[2] = w.z;
            }
            __syncthreads();
            if (tid == 0) {
                double* d = s_node + 12 * op.node + 3;
                double old[9], nw[9];
                for (int k = 0; k < 9; k++) old[k] = d[k];
                mat3_mul(q, old, nw);
                for (int k = 0; k < 9; k++) d[k] = mv.f32 ? rf32(nw[k]) : nw[k];
            }
            __syncthreads();
            continue;
        }
        // translations of a subtree: TRANSLATE (offset = param), TRANSLATE_TO (param - position(node)), PIVOT ((R v) - v)
        V3 off;
        if (op.kind == BMO_KIN_TRANSLATE) off = mk3(q[0], q[1], q[2]);
        else {
            const double* pa = s_node + 12 * nd.pos_ref;
            if (op.kind == BMO_KIN_TRANSLATE_TO) off = mk3(q[0] - pa[0], q[1] - pa[1], q[2] - pa[2]);
            else {
                const double* pb = s_node + 12 * P.nodes[op.pivot].pos_ref;
                const V3 v = mk3(pa[0] - pb[0], pa[1] - pb[1], pa[2] - pb[2]);
                const V3 rv = mat3_vec(q, v);
                off = mk3(rv.x - v.x, rv.y - v.y, rv.z - v.z);
            }
        }
        __syncthreads();   // every thread has read the positions the offset depends on
        for (int j = op.node + tid; j < op.node + nd.size; j += PBLOCK) {
            double* pp = s_node + 12 * j;
            const bmo_kin_node& nj = P.nodes[j];
            const bool f32 = nj.kind == BMO_KIN_MESH && P.meshes[nj.index].f32;
            pp[0] = pp[0] + off.x; pp[1] = pp[1] + off.y; pp[2] = pp[2] + off.z;
            if (f32) { pp[0] = rf32(pp[0]); pp[1] = rf32(pp[1]); pp[2] = rf32(pp[2]); }
        }
        for (int j = op.node; j < op.node + nd.size; j++) {
            const bmo_kin_node& nj = P.nodes[j];
            if (nj.kind != BMO_KIN_MESH) continue;
            const MeshView mv = P.meshes[nj.index];
            for (int64_t i = tid; i < mv.n_vertices; i += PBLOCK) {
                double* v = verts + 3 * (mv.first_vertex + i);
                V3 w = mk3(v[0] + off.x, v[1] + off.y, v[2] + off.z);
                if (mv.f32) w = mk3(rf32(w.x), rf32(w.y), rf32(w.z));
                v[0] = w.x; v[1] = w.y; v[2] = w.z;
            }
        }
        __syncthreads();
    }

    // ---- this pose's tables ----
    bmo_prim* prims = P.prims + (size_t)pose * P.n_prims;
    for (int i = tid; i < P.n_prims; i += PBLOCK) prims[i] = P.prims0[i];
    double* dp = P.detpose + (size_t)pose * 12 * P.n_objects;
    for (int k = tid; k < 12 * P.n_objects; k += PBLOCK) dp[k] = P.detpose0[k];
    __syncthreads();
    for (int j = tid; j < P.n_nodes; j += PBLOCK) {
        const bmo_kin_node& nd = P.nodes[j];
        const double* s = s_node + 12 * j;
        if (nd.kind == BMO_KIN_PRIM) {
            bmo_prim& pr = prims[nd.index];
            pr.pos[0] = s[0]; pr.pos[1] = s[1]; pr.pos[2] = s[2];
            bool ident = true;
#pragma unroll
            for (int a = 0; a < 3; a++)
#pragma unroll
                for (int b = 0; b < 3; b++) {
                    const double v = s[3 + 3 * b + a];           // transposed_dir = transpose(dir)
                    pr.tdir[3 * a + b] = v;
                    ident = ident && v == (a == b ? 1.0 : 0.0);
                }
            pr.reserved = (pr.reserved & ~1) | (ident ? 1 : 0);  // bit 0: identity orientation (w2s_f), bit 1 kept
        }
        if (nd.object >= 0) {
            double* d = dp + 12 * nd.object;
            for (int k = 0; k < 12; k++) d[k] = s[k];
        }
    }
    __syncthreads();

    // ---- part bounds: enclosing sphere + axis-aligned box, inflated like the flattener does ----
    double* bnd = P.bounds + (size_t)pose * NBOUND * P.n_parts;
    for (int p = 0; p < P.n_parts; p++) {
        const bmo_part& pt = P.parts[p];
        if (pt.shape_kind == BMO_SHAPE_SDF) {
            if (tid != 0) continue;
            double c[3] = {0, 0, 0}, lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
            int nm = 0;
            for (int i = pt.first; i < pt.first + pt.count; i += (prims[i].type == BMO_PRIM_MENISCUS ? 4 : 1)) {
                const bmo_prim& pr = prims[i];
                const double* b = P.prim_bounds + 10 * i;
                // world = pos + dir * local, dir = transpose(tdir)
                for (int k = 0; k < 3; k++) c[k] += pr.pos[k] + (pr.tdir[k] * b[0] + pr.tdir[3 + k] * b[1] + pr.tdir[6 + k] * b[2]);
                for (int corner = 0; corner < 8; corner++) {
                    const double x = (corner & 4) ? b[7] : b[4], y = (corner & 2) ? b[8] : b[5], z = (corner & 1) ? b[9] : b[6];
                    for (int k = 0; k < 3; k++) {
                        const double w = pr.pos[k] + (pr.tdir[k] * x + pr.tdir[3 + k] * y + pr.tdir[6 + k] * z);
                        lo[k] = fmin(lo[k], w); hi[k] = fmax(hi[k], w);
                    }
                }
                nm++;
            }
            for (int k = 0; k < 3; k++) c[k] /= nm;
            double r = 0;
            for (int i = pt.first; i < pt.first + pt.count; i += (prims[i].type == BMO_PRIM_MENISCUS ? 4 : 1)) {
                const bmo_prim& pr = prims[i];
                const double* b = P.prim_bounds + 10 * i;
                double d2 = 0;
                for (int k = 0; k < 3; k++) {
                    const double w = pr.pos[k] + (pr.tdir[k] * b[0] + pr.tdir[3 + k] * b[1] + pr.tdir[6 + k] * b[2]) - c[k];
                    d2 += w * w;
                }
                r = fmax(r, sqrt(d2) + b[3]);
            }
            double* o = bnd + NBOUND * p;
            o[0] = c[0]; o[1] = c[1]; o[2] = c[2]; o[3] = r * (1 + 2 * P.bound_rel) + P.bound_abs;
            for (int k = 0; k < 3; k++) {
                const double pad = P.bound_abs + 2 * P.bound_rel * fmax(fabs(lo[k]), fabs(hi[k]));
                o[4 + k] = lo[k] - pad; o[7 + k] = hi[k] + pad;
            }
        } else {   // mesh: centre = mean of the vertices, radius = farthest vertex, box = min / max (block-wide reductions)
            const MeshView mv = P.meshes[pt.first];
            const double* v = verts + 3 * mv.first_vertex;
            double acc[7] = {0, 0, 0, INFINITY, INFINITY, INFINITY, 0};
            double mx[3] = {-INFINITY, -INFINITY, -INFINITY};
            for (int64_t i = tid; i < mv.n_vertices; i += PBLOCK)
                for (int k = 0; k < 3; k++) { const double w = v[3 * i + k]; acc[k] += w; acc[3 + k] = fmin(acc[3 + k], w); mx[k] = fmax(mx[k], w); }
            double c[3], lo[3], hi[3];
            for (int k = 0; k < 3; k++) {
                double a = acc[k], l = acc[3 + k], h = mx[k];
                for (int s = 16; s > 0; s >>= 1) {
                    a += __shfl_xor_sync(0xffffffffu, a, s);
                    l = fmin(l, __shfl_xor_sync(0xffffffffu, l, s));
                    h = fmax(h, __shfl_xor_sync(0xffffffffu, h, s));
                }
                __syncthreads();
                if ((tid & 31) == 0) { s_red[tid >> 5][0] = a; s_red[tid >> 5][1] = l; s_red[tid >> 5][2] = h; }
                __syncthreads();
                a = 0; l = INFINITY; h = -INFINITY;
                for (int w = 0; w < PBLOCK / 32; w++) { a += s_red[w][0]; l = fmin(l, s_red[w][1]); h = fmax(h, s_red[w][2]); }
                c[k] = a / (double)mv.n_vertices; lo[k] = l; hi[k] = h;
            }
            double r2 = 0;
            for (int64_t i = tid; i < mv.n_vertices; i += PBLOCK) {
                double d2 = 0;
                for (int k = 0; k < 3; k++) { const double w = v[3 * i + k] - c[k]; d2 += w * w; }
                r2 = fmax(r2, d2);
            }
            for (int s = 16; s > 0; s >>= 1) r2 = fmax(r2, __shfl_xor_sync(0xffffffffu, r2, s));
            __syncthreads();
            if ((tid & 31) == 0) s_red[tid >> 5][3] = r2;
            __syncthreads();
            if (tid == 0) {
                r2 = 0;
                for (int w = 0; w < PBLOCK / 32; w++) r2 = fmax(r2, s_red[w][3]);
                double* o = bnd + NBOUND * p;
                o[0] = c[0]; o[1] = c[1]; o[2] = c[2]; o[3] = sqrt(r2) * (1 + 2 * P.bound_rel) + P.bound_abs;
                for (int k = 0; k < 3; k++) {
                    const double pad = P.bound_abs + 2 * P.bound_rel * fmax(fabs(lo[k]), fabs(hi[k]));
                    o[4 + k] = lo[k] - pad; o[7 + k] = hi[k] + pad;
                }
            }
        }
    }
}

}  // namespace bmo

int32_t bmo_system_set_kinematics(bmo_sys* s, int32_t n_nodes, const bmo_kin_node* nodes, const double* prim_bounds) {
    if (!s || n_nodes < 1 || !nodes || (!prim_bounds && !s->prims.empty())) return fail(BMO_EINVAL, "bmo_system_set_kinematics: bad arguments");
    const int n_prims = (int)s->prims.size(), n_meshes = (int)s->meshes.size(), n_objects = (int)s->objects.size();
    std::vector<char> prim_seen((size_t)std::max(n_prims, 1), 0), mesh_seen((size_t)std::max(n_meshes, 1), 0);
    for (int i = 0; i < n_nodes; i++) {
        const bmo_kin_node& nd = nodes[i];
        if (nd.kind < BMO_KIN_GROUP || nd.kind > BMO_KIN_MESH) return fail(BMO_EINVAL, "kinematic node: unknown kind");
        if (nd.size < 1 || i + nd.size > n_nodes) return fail(BMO_EINVAL, "kinematic node: subtree leaves the table");
        if (nd.pos_ref < 0 || nd.pos_ref >= n_nodes) return fail(BMO_EINVAL, "kinematic node: pos_ref out of range");
        if (nodes[nd.pos_ref].kind == BMO_KIN_MULTI) return fail(BMO_EINVAL, "kinematic node: pos_ref must name a node with its own position");
        if (nd.object >= n_objects) return fail(BMO_EINVAL, "kinematic node: object out of range");
        if (nd.kind == BMO_KIN_PRIM) {
            if (nd.index < 0 || nd.index >= n_prims || prim_seen[nd.index]) return fail(BMO_EINVAL, "kinematic node: bad prim index");
            prim_seen[nd.index] = 1;
            if (nd.size != 1) return fail(BMO_EINVAL, "kinematic node: a prim is a leaf");
        }
        if (nd.kind == BMO_KIN_MESH) {
            if (nd.index < 0 || nd.index >= n_meshes || mesh_seen[nd.index]) return fail(BMO_EINVAL, "kinematic node: bad mesh index");
            mesh_seen[nd.index] = 1;
            if (nd.size != 1) return fail(BMO_EINVAL, "kinematic node: a mesh is a leaf");
        }
    }
    // every top-level prim record and every mesh must be driven by a node (meniscus children follow their frame)
    for (const bmo_part& pt : s->parts) {
        if (pt.shape_kind == BMO_SHAPE_MESH) { if (!mesh_seen[pt.first]) return fail(BMO_EINVAL, "bmo_system_set_kinematics: a mesh has no node"); }
        else for (int i = pt.first; i < pt.first + pt.count; i += (s->prims[i].type == BMO_PRIM_MENISCUS ? 4 : 1))
            if (!prim_seen[i]) return fail(BMO_EINVAL, "bmo_system_set_kinematics: a primitive has no node");
    }
    BMO_CUDA(cudaSetDevice(s->ctx->device));
    BMO_CUDA(cudaStreamSynchronize(s->ctx->stream));
    // the new tables replace the live ones only once all of them are on the device
    DevTable<bmo_kin_node> d_kin_nodes; DevTable<double> d_prim_bounds; DevTable<bmo_prim> d_prims0; DevTable<double> d_vertices0, d_detpose0;
    int32_t rc;
    if ((rc = upload(d_kin_nodes, nodes, (size_t)n_nodes))) return rc;
    if ((rc = upload(d_prim_bounds, prim_bounds, (size_t)10 * n_prims))) return rc;
    if ((rc = upload(d_prims0, s->prims.data(), s->prims.size()))) return rc;
    if ((rc = upload(d_vertices0, s->h_vertices.data(), s->h_vertices.size()))) return rc;
    if ((rc = upload(d_detpose0, s->h_detpose.data(), s->h_detpose.size()))) return rc;
    s->kin_nodes.assign(nodes, nodes + n_nodes);
    s->d_kin_nodes = std::move(d_kin_nodes); s->d_prim_bounds = std::move(d_prim_bounds); s->d_prims0 = std::move(d_prims0);
    s->d_vertices0 = std::move(d_vertices0); s->d_detpose0 = std::move(d_detpose0);
    return BMO_OK;
}

int32_t bmo_system_apply_poses(bmo_sys* s, int32_t n_poses, int32_t n_ops, const bmo_kin_op* ops, int32_t n_params, const double* params) {
    NvtxRange nvtx_("bmo_system_apply_poses");
    if (!s || n_poses < 1 || n_ops < 0 || n_params < 0 || (n_ops > 0 && !ops) || (n_params > 0 && !params))
        return fail(BMO_EINVAL, "bmo_system_apply_poses: bad arguments");
    if (s->kin_nodes.empty()) return fail(BMO_ESTATE, "bmo_system_apply_poses: call bmo_system_set_kinematics first");
    const int n_nodes = (int)s->kin_nodes.size();
    bool mesh_with_bvh_moves = false;
    for (int o = 0; o < n_ops; o++) {
        const bmo_kin_op& op = ops[o];
        if (op.kind < BMO_KIN_TRANSLATE || op.kind > BMO_KIN_PIVOT) return fail(BMO_EINVAL, "kinematic op: unknown kind");
        if (op.node < 0 || op.node >= n_nodes) return fail(BMO_EINVAL, "kinematic op: node out of range");
        if (op.kind == BMO_KIN_PIVOT && (op.pivot < 0 || op.pivot >= n_nodes)) return fail(BMO_EINVAL, "kinematic op: pivot out of range");
        if (op.param < 0 || op.param >= n_params) return fail(BMO_EINVAL, "kinematic op: param out of range");
        const bmo_kin_node& nd = s->kin_nodes[op.node];
        if (op.kind == BMO_KIN_ROT_FRAME && !(nd.kind == BMO_KIN_GROUP || nd.kind == BMO_KIN_UNION)) return fail(BMO_EINVAL, "ROT_FRAME needs a GROUP or UNION node");
        if (op.kind == BMO_KIN_ROT_LEAF && !(nd.kind == BMO_KIN_PRIM || nd.kind == BMO_KIN_MESH)) return fail(BMO_EINVAL, "ROT_LEAF needs a PRIM or MESH node");
        if (op.kind != BMO_KIN_ROT_FRAME)
            for (int j = op.node; j < op.node + nd.size; j++)
                if (s->kin_nodes[j].kind == BMO_KIN_MESH && s->meshes[s->kin_nodes[j].index].n_nodes > 0) mesh_with_bvh_moves = true;
    }
    const size_t smem = (size_t)n_nodes * 12 * sizeof(double);
    if (smem > 200 * 1024) return fail(BMO_EINVAL, "bmo_system_apply_poses: kinematic tree too large for one block's shared memory");
    bmo_ctx* ctx = s->ctx;
    BMO_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    BMO_CUDA(cudaStreamSynchronize(st));
    const size_t np = (size_t)n_poses, n_prims = s->prims.size(), n_parts = s->parts.size(), n_objects = s->objects.size();
    // the kernel writes new tables; they replace the live ones only once it has run
    DevTable<bmo_prim> d_prims; DevTable<double> d_vertices, d_bounds, d_detpose;
    int32_t rc;
    if ((rc = upload(d_prims, (const bmo_prim*)nullptr, np * n_prims))) return rc;
    if ((rc = upload(d_vertices, (const double*)nullptr, np * 3 * (size_t)s->n_vertices))) return rc;
    if ((rc = upload(d_bounds, (const double*)nullptr, np * NBOUND * n_parts))) return rc;
    if ((rc = upload(d_detpose, (const double*)nullptr, np * 12 * n_objects))) return rc;
    DevBuf<bmo_kin_op> d_ops;
    DevBuf<double> d_par;
    BMO_CUDA(d_ops.alloc((size_t)n_ops, st));
    BMO_CUDA(d_par.alloc(np * n_params * 9, st));
    if (n_ops) BMO_CUDA(cudaMemcpyAsync(d_ops.get(), ops, (size_t)n_ops * sizeof(bmo_kin_op), cudaMemcpyHostToDevice, st));
    if (n_params) BMO_CUDA(cudaMemcpyAsync(d_par.get(), params, np * n_params * 9 * sizeof(double), cudaMemcpyHostToDevice, st));
    PoseParams P{};
    P.nodes = s->d_kin_nodes.get(); P.n_nodes = n_nodes; P.ops = d_ops.get(); P.n_ops = n_ops; P.params = d_par.get(); P.n_params = n_params;
    P.prims0 = s->d_prims0.get(); P.n_prims = (int32_t)n_prims; P.parts = s->d_parts.get(); P.n_parts = (int32_t)n_parts;
    P.meshes = s->d_meshes.get(); P.n_meshes = (int32_t)s->meshes.size(); P.vertices0 = s->d_vertices0.get(); P.n_vertices = s->n_vertices;
    P.detpose0 = s->d_detpose0.get(); P.n_objects = (int32_t)n_objects; P.prim_bounds = s->d_prim_bounds.get();
    P.prims = d_prims.get(); P.vertices = d_vertices.get(); P.bounds = d_bounds.get(); P.detpose = d_detpose.get();
    P.bound_rel = 1e-9; P.bound_abs = 1e-6;   // flatten.py BOUND_REL / BOUND_ABS
    if (smem > 48 * 1024) BMO_CUDA(cudaFuncSetAttribute(apply_poses_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    apply_poses_kernel<<<(unsigned)n_poses, PBLOCK, smem, st>>>(P);
    BMO_LAUNCH(ctx, "apply_poses_kernel");
    BMO_CUDA(cudaStreamSynchronize(st));
    s->d_prims = std::move(d_prims); s->d_vertices = std::move(d_vertices); s->d_bounds = std::move(d_bounds); s->d_detpose = std::move(d_detpose);
    SysView& v = s->view;
    v.prims = s->d_prims.get(); v.vertices = s->d_vertices.get(); v.bounds = s->d_bounds.get(); v.det_pose = s->d_detpose.get();
    v.n_poses = n_poses;
    v.bvh_ok = mesh_with_bvh_moves ? 0 : 1;
    return BMO_OK;
}

int32_t bmo_system_get_pose(bmo_sys* s, int32_t pose, bmo_prim* prims, double* vertices, double* bounds, double* det_pose) {
    if (!s || pose < 0 || pose >= s->view.n_poses) return fail(BMO_EINVAL, "bmo_system_get_pose: pose out of range");
    BMO_CUDA(cudaSetDevice(s->ctx->device));
    BMO_CUDA(cudaStreamSynchronize(s->ctx->stream));
    const size_t n_prims = s->prims.size(), n_parts = s->parts.size(), n_objects = s->objects.size(), p = (size_t)pose;
    if (prims && n_prims) BMO_CUDA(cudaMemcpy(prims, s->d_prims.get() + p * n_prims, n_prims * sizeof(bmo_prim), cudaMemcpyDeviceToHost));
    if (vertices && s->n_vertices) BMO_CUDA(cudaMemcpy(vertices, s->d_vertices.get() + p * 3 * s->n_vertices, (size_t)3 * s->n_vertices * sizeof(double), cudaMemcpyDeviceToHost));
    if (bounds) BMO_CUDA(cudaMemcpy(bounds, s->d_bounds.get() + p * NBOUND * n_parts, NBOUND * n_parts * sizeof(double), cudaMemcpyDeviceToHost));
    if (det_pose) BMO_CUDA(cudaMemcpy(det_pose, s->d_detpose.get() + p * 12 * n_objects, 12 * n_objects * sizeof(double), cudaMemcpyDeviceToHost));
    return BMO_OK;
}
