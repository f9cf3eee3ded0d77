// scene.cpp — the C-ABI of include/rtb200.h: scene DAG recording, depth-first leaf numbering,
// flattening into the device layout of rt_types.h, BVH build, upload, and the render / trace entry
// points that launch the sm_100a kernels.  No CPU fallback: without a CUDA device commit / render /
// trace return RT_ERR_CUDA.
#include <cuda_runtime.h>

#include <cfloat>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <condition_variable>
#include <cstring>
#include <map>
#include <memory>
#include <string>
#include <mutex>
#include <system_error>
#include <thread>
#include <vector>

#include "../../../include/rtb200.h"
#include "../cuda/kernels.h"
#include "../rt_types.h"
#include "bvh_build.hpp"
#include "bvh_wide.hpp"
#include "io.hpp"
#include "world.hpp"

using namespace rtb;

namespace {

thread_local std::string g_err;
int32_t fail(int32_t code, const std::string& msg) {
    g_err = msg;
    return code;
}
int32_t fail_cuda(cudaError_t e, const char* what) {
    g_err = std::string(what) + ": " + cudaGetErrorString(e);
    return RT_ERR_CUDA;
}

enum NodeKind { N_SPHERE, N_MOVING, N_GRAVITY, N_RECT, N_BOX, N_TRI, N_MESH, N_LIST, N_BVH, N_TRANSLATE, N_ROTY, N_MEDIUM };

struct MeshData {
    std::vector<double> verts;   // xyz
    std::vector<uint32_t> faces; // 3 per triangle
};

struct Node {
    NodeKind kind;
    double d[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    int32_t axis = 0;
    int32_t mat = -1;
    std::vector<int32_t> children;
    std::shared_ptr<MeshData> mesh;
    std::shared_ptr<std::vector<double>> grav; // GravitySphere::stored
    int32_t prim_base = -1;                    // depth-first id of the first leaf this node produces
};

struct TexDesc {
    uint32_t type;
    double rgb[3] = {0, 0, 0};
    int32_t a = 0, b = 0;
    double scale = 0;
    int32_t w = 0, h = 0;
    std::shared_ptr<PerlinTable> perlin;
    std::shared_ptr<std::vector<float>> texels; // rgba
};
struct MatDesc {
    uint32_t type;
    int32_t tex = 0;
    double albedo[3] = {0, 0, 0};
    double param = 0;
};

struct CameraDesc {
    bool set = false;
    DCamera cam;
};

struct DeviceBuffers { // one grow-only device arena + one pinned staging buffer: a commit is ONE H2D copy
    char* arena = nullptr;
    size_t capacity = 0;
    char* staging = nullptr;
    size_t staging_capacity = 0;
    DeviceScene scene;
    bool valid = false;
    int device = 0;   // CUDA device the arena lives on (the device current at rt_scene_commit)
    size_t bytes = 0; // bytes uploaded by the last commit
    uint64_t generation = 0; // bumped by every commit: replicas on other GPUs (rt_render_multi) compare it
    // (offset of a pointer field inside DeviceScene, offset of its array inside the arena / staging buffer): lets a replica on
    // another GPU re-base the same flattened bytes without running the flattener again
    std::vector<std::pair<size_t, size_t>> layout;
    int64_t device_built_prims = 0; // primitives whose BVH the last commit built on the device (lbvh.cu)
    float device_build_ms = 0.f;
    void release() {
        if (arena) cudaFree(arena);
        if (staging) cudaFreeHost(staging);
        arena = nullptr; staging = nullptr; capacity = 0; staging_capacity = 0;
        valid = false;
    }
};

// Output side of rt_render / rt_render_multi, kept between calls (no cudaMalloc / cudaFree / pageable staging per render):
// the accumulator and the byte Screen on the gathering GPU, one pinned host mirror of the byte Screen.
struct RenderBuffers {
    int64_t* d_accum = nullptr;
    uint8_t* d_u8 = nullptr;
    uint8_t* h_u8 = nullptr; // pinned
    size_t cap = 0;          // elements (W * H * 3)
    cudaStream_t stream = nullptr;
    void release() {
        if (d_accum) cudaFree(d_accum);
        if (d_u8) cudaFree(d_u8);
        if (h_u8) cudaFreeHost(h_u8);
        if (stream) cudaStreamDestroy(stream);
        d_accum = nullptr; d_u8 = nullptr; h_u8 = nullptr; stream = nullptr; cap = 0;
    }
};

// Working set of rt_render_adaptive, kept between calls like RenderBuffers: the half accumulators A and B, the active pixel list and
// the next one, per-pixel sample counts, the convergence mask, the compaction flags and CUB's temp storage; the pinned count word the
// host reads once per check point.
struct AdaptiveBuffers {
    int64_t* d_a = nullptr;
    int64_t* d_b = nullptr;
    uint32_t* d_list[2] = {nullptr, nullptr};
    int32_t* d_samples = nullptr;
    uint8_t* d_u = nullptr;
    uint8_t* d_keep = nullptr;
    void* d_temp = nullptr;
    size_t temp_bytes = 0;
    uint32_t* h_count = nullptr; // pinned
    size_t cap = 0;              // pixels (W * H)
    void release() {
        if (d_a) cudaFree(d_a);
        if (d_b) cudaFree(d_b);
        for (uint32_t*& l : d_list) { if (l) cudaFree(l); l = nullptr; }
        if (d_samples) cudaFree(d_samples);
        if (d_u) cudaFree(d_u);
        if (d_keep) cudaFree(d_keep);
        if (d_temp) cudaFree(d_temp);
        if (h_count) cudaFreeHost(h_count);
        d_a = d_b = nullptr; d_samples = nullptr; d_u = d_keep = nullptr; d_temp = nullptr; temp_bytes = 0; h_count = nullptr; cap = 0;
    }
};

// The committed scene on one more GPU (rt_render_multi): same flattened bytes, pointers re-based into this GPU's arena.
struct Replica {
    int device = -1;
    char* arena = nullptr;
    size_t capacity = 0;
    uint64_t generation = ~0ull;
    DeviceScene scene;
    Workspace* workspace = nullptr;
    int64_t* d_accum = nullptr; // rt_render_multi's shard; rt_render_adaptive_multi's half accumulators A | B (B at an even offset)
    size_t accum_cap = 0;
    uint32_t* d_list = nullptr; // rt_render_adaptive_multi: this GPU's copy of the active pixel list
    size_t list_cap = 0;
    cudaStream_t stream = nullptr;
    bool peer_ok = false; // the gathering GPU can read this arena's accumulator directly
    int64_t* d_stage = nullptr; // on the gathering GPU, only when peer access is unavailable
    size_t stage_cap = 0;
    void release() {
        int cur = 0;
        cudaGetDevice(&cur);
        if (device >= 0) cudaSetDevice(device);
        if (arena) cudaFree(arena);
        if (d_accum) cudaFree(d_accum);
        if (d_list) cudaFree(d_list);
        if (stream) cudaStreamDestroy(stream);
        free_workspace(workspace);
        cudaSetDevice(cur);
        if (d_stage) cudaFree(d_stage);
        arena = nullptr; d_accum = nullptr; d_list = nullptr; stream = nullptr; workspace = nullptr; d_stage = nullptr;
        accum_cap = list_cap = stage_cap = 0;
    }
};

} // namespace

struct rt_scene {
    std::vector<TexDesc> tex;
    std::vector<MatDesc> mats;
    std::vector<Node> nodes;
    int32_t root = -1;
    CameraDesc camera;
    double background[3] = {0, 0, 0};
    double background_top[3] = {0, 0, 0};
    bool bg_gradient = false;
    int32_t n_prims = 0;
    bool committed = false;
    double span0 = 0.0, span1 = 1.0; // time span the moving-primitive bounds cover
    double domain_radius = 0.0;
    DeviceBuffers dev;
    RenderTuning tuning;
    Workspace* workspace = nullptr;
    RenderBuffers out;
    AdaptiveBuffers adaptive;
    std::vector<Replica> replicas; // GPUs 1 .. n-1 of rt_render_multi (GPU 0 is `dev`)
    std::shared_ptr<void> debug_flat; // rt_debug_host_scene: the host-flattened arrays handed to the caller
    ~rt_scene() {
        for (Replica& r : replicas) r.release();
        out.release();
        adaptive.release();
        dev.release();
        free_workspace(workspace);
    }
};

#define CHECK_SCENE(s) \
    if (!(s)) return fail(RT_ERR_INVALID, "null scene")
#define CHECK_TEX(s, id) \
    if ((id) < 0 || (size_t)(id) >= (s)->tex.size()) return fail(RT_ERR_INVALID, "texture id out of range")
#define CHECK_MAT(s, id) \
    if ((id) < 0 || (size_t)(id) >= (s)->mats.size()) return fail(RT_ERR_INVALID, "material id out of range")
#define CHECK_OBJ(s, id) \
    if ((id) < 0 || (size_t)(id) >= (s)->nodes.size()) return fail(RT_ERR_INVALID, "hittable id out of range")

namespace {

int32_t add_node(rt_scene* s, Node&& n) {
    s->nodes.push_back(std::move(n));
    s->committed = false;
    return (int32_t)s->nodes.size() - 1;
}

// ---------------------------------------------------------------- depth-first leaf numbering
// Same walk as the oracle's number_leaves(): leaves get ids at first visit; a box takes 6, a mesh
// one per triangle, a medium takes one id and then numbers its boundary.
void number_leaves(rt_scene* s, int32_t id, int32_t& next) {
    Node& n = s->nodes[(size_t)id];
    switch (n.kind) {
    case N_SPHERE: case N_MOVING: case N_GRAVITY: case N_RECT: case N_TRI:
        if (n.prim_base < 0) { n.prim_base = next; next += 1; }
        break;
    case N_BOX:
        if (n.prim_base < 0) { n.prim_base = next; next += 6; }
        break;
    case N_MESH:
        if (n.prim_base < 0) { n.prim_base = next; next += (int32_t)(n.mesh->faces.size() / 3); }
        break;
    case N_LIST: case N_BVH: case N_TRANSLATE: case N_ROTY:
        for (int32_t c : n.children) number_leaves(s, c, next);
        break;
    case N_MEDIUM:
        if (n.prim_base < 0) { n.prim_base = next; next += 1; }
        number_leaves(s, n.children[0], next);
        break;
    }
}

// ---------------------------------------------------------------- flattening
// Mesh-sized host loops (871 200 triangles: boxes, build records, typed triangles) run in contiguous chunks on up to 16 threads;
// every index is written by exactly one thread, so the arrays are those of the serial loop.
template <class F> void parallel_chunks(size_t n, F&& body) {
    const unsigned hw = std::thread::hardware_concurrency();
    const size_t threads = n >= 65536 ? std::min<size_t>(16, std::max(1u, hw)) : 1;
    if (threads <= 1) { body((size_t)0, n); return; }
    const size_t chunk = (n + threads - 1) / threads;
    std::vector<std::thread> pool;
    for (size_t t = 1; t < threads; ++t) {
        const size_t b = std::min(n, t * chunk), e = std::min(n, b + chunk);
        if (b < e) pool.emplace_back([&body, b, e]() { body(b, e); });
    }
    body((size_t)0, std::min(n, chunk));
    for (std::thread& th : pool) th.join();
}

struct FlatPrim {
    uint32_t type;
    int32_t node;     // source node
    uint32_t sub;     // triangle index inside a mesh
    uint32_t mat, prim_id;
    double bmin[3], bmax[3];
};
struct InstBuild {
    std::vector<int32_t> key; // transform node ids, outermost first
    std::vector<XformOp> chain;
    std::vector<FlatPrim> prims;
};
struct WorldBuild {
    std::vector<InstBuild> inst;
};
struct MediumBuild {
    int32_t node;
    std::vector<XformOp> chain;
    size_t world;
};

struct Flattener {
    rt_scene* s;
    std::vector<WorldBuild> worlds;
    std::vector<MediumBuild> media;
    std::string error;
    int32_t status = RT_OK;

    InstBuild& instance_for(size_t world, const std::vector<int32_t>& key, const std::vector<XformOp>& chain) {
        for (InstBuild& ib : worlds[world].inst)
            if (ib.key == key) return ib;
        InstBuild ib;
        ib.key = key;
        ib.chain = chain;
        worlds[world].inst.push_back(std::move(ib));
        return worlds[world].inst.back();
    }

    void sphere_box(const double c[3], double r, double mn[3], double mx[3]) {
        for (int a = 0; a < 3; ++a) { mn[a] = c[a] - std::fabs(r); mx[a] = c[a] + std::fabs(r); }
    }

    void add_leaf(size_t world, const std::vector<int32_t>& key, const std::vector<XformOp>& chain, int32_t id) {
        const Node& n = s->nodes[(size_t)id];
        InstBuild& ib = instance_for(world, key, chain);
        FlatPrim p;
        p.node = id; p.sub = 0; p.mat = (uint32_t)n.mat; p.prim_id = (uint32_t)n.prim_base;
        switch (n.kind) {
        case N_SPHERE: p.type = PRIM_SPHERE; sphere_box(n.d, n.d[3], p.bmin, p.bmax); break;
        case N_MOVING: { // bounds over the span (MovingSphere::bounding_box, hit.rs:317-327; motion is linear)
            p.type = PRIM_MOVING;
            const double t0 = n.d[6], t1 = n.d[7], r = n.d[8];
            double c0[3], c1[3], a0[3], a1[3], b0[3], b1[3];
            for (int a = 0; a < 3; ++a) {
                c0[a] = n.d[a] + ((s->span0 - t0) / (t1 - t0)) * (n.d[3 + a] - n.d[a]);
                c1[a] = n.d[a] + ((s->span1 - t0) / (t1 - t0)) * (n.d[3 + a] - n.d[a]);
            }
            sphere_box(c0, r, a0, a1);
            sphere_box(c1, r, b0, b1);
            for (int a = 0; a < 3; ++a) { p.bmin[a] = std::fmin(a0[a], b0[a]); p.bmax[a] = std::fmax(a1[a], b1[a]); }
        } break;
        case N_GRAVITY: { // bounds over the uploaded window of the height table
            p.type = PRIM_GRAVITY;
            int64_t i0, i1;
            gravity_window(*n.grav, i0, i1);
            double ymin = 1e300, ymax = -1e300;
            for (int64_t i = i0; i <= i1; ++i) { ymin = std::fmin(ymin, (*n.grav)[(size_t)i]); ymax = std::fmax(ymax, (*n.grav)[(size_t)i]); }
            const double r = std::fabs(n.d[4]);
            p.bmin[0] = n.d[0] - r; p.bmax[0] = n.d[0] + r;
            p.bmin[1] = ymin - r; p.bmax[1] = ymax + r;
            p.bmin[2] = n.d[2] - r; p.bmax[2] = n.d[2] + r;
        } break;
        case N_RECT: { // hit.rs:503-508, 568-573, 633-638
            p.type = PRIM_RECT;
            const int ax = n.axis, ia = ax == 0 ? 1 : 0, ib2 = ax == 2 ? 1 : 2;
            p.bmin[ax] = n.d[4] - 0.0001; p.bmax[ax] = n.d[4] + 0.0001;
            p.bmin[ia] = std::fmin(n.d[0], n.d[1]); p.bmax[ia] = std::fmax(n.d[0], n.d[1]);
            p.bmin[ib2] = std::fmin(n.d[2], n.d[3]); p.bmax[ib2] = std::fmax(n.d[2], n.d[3]);
        } break;
        case N_BOX:
            p.type = PRIM_BOX;
            for (int a = 0; a < 3; ++a) { p.bmin[a] = std::fmin(n.d[a], n.d[3 + a]); p.bmax[a] = std::fmax(n.d[a], n.d[3 + a]); }
            break;
        case N_TRI:
            p.type = PRIM_TRI;
            for (int a = 0; a < 3; ++a) {
                p.bmin[a] = std::fmin(n.d[a], std::fmin(n.d[3 + a], n.d[6 + a]));
                p.bmax[a] = std::fmax(n.d[a], std::fmax(n.d[3 + a], n.d[6 + a]));
            }
            break;
        case N_MESH: {
            const MeshData& m = *n.mesh;
            const size_t nt = m.faces.size() / 3, base = ib.prims.size();
            ib.prims.resize(base + nt);
            FlatPrim* out = ib.prims.data() + base;
            const int32_t mat = n.mat, prim_base = n.prim_base;
            parallel_chunks(nt, [&m, out, id, mat, prim_base](size_t t0, size_t t1) {
                for (size_t t = t0; t < t1; ++t) {
                    FlatPrim q;
                    q.type = PRIM_TRI; q.node = id; q.sub = (uint32_t)t; q.mat = (uint32_t)mat; q.prim_id = (uint32_t)prim_base + (uint32_t)t;
                    const double* v0 = &m.verts[3 * (size_t)m.faces[3 * t]];
                    const double* v1 = &m.verts[3 * (size_t)m.faces[3 * t + 1]];
                    const double* v2 = &m.verts[3 * (size_t)m.faces[3 * t + 2]];
                    for (int a = 0; a < 3; ++a) {
                        q.bmin[a] = std::fmin(v0[a], std::fmin(v1[a], v2[a]));
                        q.bmax[a] = std::fmax(v0[a], std::fmax(v1[a], v2[a]));
                    }
                    out[t] = q;
                }
            });
            return;
        }
        default: return;
        }
        ib.prims.push_back(p);
    }

    void gravity_window(const std::vector<double>& tab, int64_t& i0, int64_t& i1) {
        const double q0 = s->span0 / 0.001, q1 = s->span1 / 0.001;
        i0 = q0 > 0.0 ? (int64_t)q0 : 0;
        i1 = q1 > 0.0 ? (int64_t)q1 : 0;
        // hit.rs:373: the table answers while (time / incr) as usize + 1 <= stored.len(); past it GravitySphere::get_center re-integrates
        // with other constants (2 * radius, -0.8 bounce: hit.rs:381-393), which is not reproduced here (DESIGN.md divergence 5): refuse the
        // shutter instead of silently holding the last table entry
        if (i1 + 1 > (int64_t)tab.size() && status == RT_OK) {
            status = RT_ERR_UNSUPPORTED;
            error = "camera shutter reaches past the GravitySphere height table (time >= ~100): the reference's fallback integration (hit.rs:381-393) is not supported";
        }
        i1 += 1; // time2 itself is exclusive, one guard entry
        const int64_t last = (int64_t)tab.size() - 1;
        i0 = std::min(std::max<int64_t>(i0, 0), last);
        i1 = std::min(std::max<int64_t>(i1, i0), last);
    }

    void visit(int32_t id, size_t world, std::vector<int32_t>& key, std::vector<XformOp>& chain, bool in_boundary, int depth) {
        if (status != RT_OK) return;
        if (depth > 4096) { status = RT_ERR_UNSUPPORTED; error = "scene graph deeper than 4096 (cycle?)"; return; }
        const Node& n = s->nodes[(size_t)id];
        switch (n.kind) {
        case N_LIST: case N_BVH:
            for (int32_t c : n.children) visit(c, world, key, chain, in_boundary, depth + 1);
            break;
        case N_TRANSLATE: {
            XformOp op; op.type = XF_TRANSLATE; op.pad_ = 0; op.a = n.d[0]; op.b = n.d[1]; op.c = n.d[2];
            key.push_back(id); chain.push_back(op);
            visit(n.children[0], world, key, chain, in_boundary, depth + 1);
            key.pop_back(); chain.pop_back();
        } break;
        case N_ROTY: {
            XformOp op; op.type = XF_ROTATE_Y; op.pad_ = 0; op.a = n.d[0]; op.b = n.d[1]; op.c = 0.0; // sin, cos
            key.push_back(id); chain.push_back(op);
            visit(n.children[0], world, key, chain, in_boundary, depth + 1);
            key.pop_back(); chain.pop_back();
        } break;
        case N_MEDIUM: {
            if (in_boundary) { status = RT_ERR_UNSUPPORTED; error = "ConstantMedium inside the boundary of another ConstantMedium is not supported"; return; }
            MediumBuild mb;
            mb.node = id;
            mb.chain = chain;
            worlds.emplace_back();
            mb.world = worlds.size() - 1;
            media.push_back(mb);
            std::vector<int32_t> k2;
            std::vector<XformOp> c2;
            visit(n.children[0], mb.world, k2, c2, true, depth + 1);
        } break;
        default:
            add_leaf(world, key, chain, id);
            break;
        }
    }
};

struct UploadPlan { // collects the flattened arrays, lays them out 256-byte aligned, uploads them in one copy
    struct Piece { const void* src; size_t bytes; size_t offset; const void** dst; };
    std::vector<Piece> pieces;
    size_t total = 0;
    template <class T> void add(const std::vector<T>& v, const T*& field) {
        total = (total + 255) & ~(size_t)255;
        Piece p;
        p.src = v.data(); p.bytes = v.size() * sizeof(T); p.offset = total;
        p.dst = reinterpret_cast<const void**>(&field);
        pieces.push_back(p);
        total += std::max<size_t>(p.bytes, 16);
    }
    cudaError_t run(DeviceBuffers& dev) {
        cudaError_t e;
        if (total > dev.capacity) {
            if (dev.arena) cudaFree(dev.arena);
            dev.arena = nullptr; dev.capacity = 0;
            const size_t cap = total + total / 4 + 4096;
            if ((e = cudaMalloc(&dev.arena, cap)) != cudaSuccess) return e;
            dev.capacity = cap;
        }
        if (total > dev.staging_capacity) {
            if (dev.staging) cudaFreeHost(dev.staging);
            dev.staging = nullptr; dev.staging_capacity = 0;
            const size_t cap = total + total / 4 + 4096;
            if ((e = cudaMallocHost(&dev.staging, cap)) != cudaSuccess) return e;
            dev.staging_capacity = cap;
        }
        dev.layout.clear();
        for (const Piece& p : pieces) {
            if (p.bytes) std::memcpy(dev.staging + p.offset, p.src, p.bytes);
            *p.dst = dev.arena + p.offset;
            dev.layout.emplace_back((size_t)(reinterpret_cast<const char*>(p.dst) - reinterpret_cast<const char*>(&dev.scene)), p.offset);
        }
        if ((e = cudaMemcpy(dev.arena, dev.staging, total, cudaMemcpyHostToDevice)) != cudaSuccess) return e;
        dev.bytes = total;
        return cudaSuccess;
    }
};

bool tex_reads_uv(const rt_scene* s, int32_t t, int depth = 0) {
    if (depth > 64) return false;
    const TexDesc& d = s->tex[(size_t)t];
    if (d.type == TEX_IMAGE) return true;
    if (d.type == TEX_CHECKER) return tex_reads_uv(s, d.a, depth + 1) || tex_reads_uv(s, d.b, depth + 1);
    return false;
}

struct HostFlat {
    std::vector<BvhNode32> mnodes;     // motion-interpolated boxes (two entries per node), empty without MovingSpheres
    float device_build_ms = 0.f;      // device LBVH time (CUDA events), 0 when the host builder ran
    int64_t device_built_prims = 0;
    std::vector<BvhNode32> nodes;
    std::vector<DSphere> spheres; std::vector<DMoving> movings; std::vector<DGravity> gravities; std::vector<double> gtable;
    std::vector<DRect> rects; std::vector<DBox> boxes; std::vector<DTri> tris;
    std::vector<PrimMeta> meta[PRIM_TYPE_COUNT];
    std::vector<Instance> instances;
    std::vector<XformOp> ops;
    std::vector<Medium> media;
    std::vector<DMaterial> dmats;
    std::vector<DTexture> dtex;
    std::vector<PerlinTable> perlin;
    std::vector<float4> texels;
    uint32_t n_main_instances = 0;
    int max_depth = 0;
    double pad = 0.0;
    std::vector<float4> mnodes4;       // motion form of nodes4 (MovingSphere scenes with a 4-wide collapse)
    std::vector<float4> nodes4;        // 4-wide collapse of the single main instance's tree (tuning.bvh_wide), else empty
    uint32_t root4 = RT_WIDE_EMPTY;
    int wide_depth = 0;
};

// host half of rt_scene_commit: numbering, flattening, BVH build (no CUDA needed)
struct MotionBox { // bounds of a primitive / subtree at the two ends of the shutter
    double lo0[3], hi0[3], lo1[3], hi1[3];
    void clear() { for (int a = 0; a < 3; ++a) { lo0[a] = lo1[a] = DBL_MAX; hi0[a] = hi1[a] = -DBL_MAX; } }
    void merge(const MotionBox& o) {
        for (int a = 0; a < 3; ++a) {
            lo0[a] = std::fmin(lo0[a], o.lo0[a]); hi0[a] = std::fmax(hi0[a], o.hi0[a]);
            lo1[a] = std::fmin(lo1[a], o.lo1[a]); hi1[a] = std::fmax(hi1[a], o.hi1[a]);
        }
    }
};

struct PhaseTimer { // RTB200_COMMIT_TIMING=1: phase times of rt_scene_commit on stderr
    bool on = std::getenv("RTB200_COMMIT_TIMING") != nullptr;
    std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
    void lap(const char* what) {
        if (!on) return;
        const auto t1 = std::chrono::steady_clock::now();
        std::fprintf(stderr, "[rtb200 commit] %-22s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(t1 - t0).count());
        t0 = t1;
    }
};

int32_t flatten_host(rt_scene* s, HostFlat& HF, bool allow_device_build = false) {
    if (s->root < 0) return fail(RT_ERR_STATE, "no root set (rt_scene_set_root)");
    PhaseTimer pt;
    int32_t next = s->n_prims;
    number_leaves(s, s->root, next);
    s->n_prims = next;
    if (s->camera.set) { s->span0 = std::fmin(s->camera.cam.time1, s->camera.cam.time2); s->span1 = std::fmax(s->camera.cam.time1, s->camera.cam.time2); }
    else { s->span0 = 0.0; s->span1 = 1.0; }

    Flattener F;
    F.s = s;
    F.worlds.emplace_back();
    {
        std::vector<int32_t> key;
        std::vector<XformOp> chain;
        F.visit(s->root, 0, key, chain, false, 0);
    }
    if (F.status != RT_OK) return fail(F.status, F.error);
    pt.lap("number + visit");

    // domain radius: every coordinate the f32 slab test can see (boxes in instance space, camera origin)
    double R = 1.0;
    for (const WorldBuild& w : F.worlds)
        for (const InstBuild& ib : w.inst) {
            std::mutex mu;
            const FlatPrim* fp = ib.prims.data();
            parallel_chunks(ib.prims.size(), [&](size_t i0, size_t i1) { // a maximum: the same value in any order
                double r = 1.0;
                for (size_t i = i0; i < i1; ++i)
                    for (int a = 0; a < 3; ++a) { r = std::fmax(r, std::fabs(fp[i].bmin[a])); r = std::fmax(r, std::fabs(fp[i].bmax[a])); }
                std::lock_guard<std::mutex> lock(mu);
                R = std::fmax(R, r);
            });
        }
    if (s->camera.set)
        for (int a = 0; a < 3; ++a) R = std::fmax(R, 2.0 * std::fabs(s->camera.cam.origin[a]));
    s->domain_radius = R;

    std::vector<BvhNode32>& nodes = HF.nodes;
    std::vector<DSphere>& spheres = HF.spheres; std::vector<DMoving>& movings = HF.movings; std::vector<DGravity>& gravities = HF.gravities;
    std::vector<double>& gtable = HF.gtable;
    std::vector<DRect>& rects = HF.rects; std::vector<DBox>& boxes = HF.boxes; std::vector<DTri>& tris = HF.tris;
    std::vector<PrimMeta>* meta = HF.meta;
    std::vector<Instance>& instances = HF.instances;
    std::vector<XformOp>& ops = HF.ops;
    std::vector<Medium>& media = HF.media;
    uint32_t cursor[PRIM_TYPE_COUNT] = {0, 0, 0, 0, 0, 0};
    int& max_depth = HF.max_depth;

    BuildOptions bo;
    bo.pad = R * (1.0 / 1048576.0); // 2^-20 * R, see DESIGN.md "f32 slab conservativeness"
    HF.pad = bo.pad;
    const char* env_leaf = std::getenv("RTB200_MAX_LEAF");
    if (env_leaf) bo.max_leaf = std::max(1, std::atoi(env_leaf));
    const char* env_cp = std::getenv("RTB200_COST_PRIM");
    if (env_cp) bo.cost_prim = std::atof(env_cp);

    std::vector<MotionBox> mbox[PRIM_TYPE_COUNT];
    // the shutter-end boxes are only read by the MovingSphere refit below (96 bytes per primitive: 84 MB for the 871 200-triangle mesh)
    bool has_moving = false;
    {
        size_t per_type[PRIM_TYPE_COUNT] = {0, 0, 0, 0, 0, 0};
        for (const WorldBuild& w : F.worlds)
            for (const InstBuild& ib : w.inst)
                for (const FlatPrim& p : ib.prims) ++per_type[p.type];
        has_moving = per_type[PRIM_MOVING] != 0;
        spheres.reserve(per_type[PRIM_SPHERE]); movings.reserve(per_type[PRIM_MOVING]); gravities.reserve(per_type[PRIM_GRAVITY]);
        rects.reserve(per_type[PRIM_RECT]); boxes.reserve(per_type[PRIM_BOX]); tris.reserve(per_type[PRIM_TRI]);
        for (int t = 0; t < (int)PRIM_TYPE_COUNT; ++t) { meta[t].reserve(per_type[t]); if (has_moving) mbox[t].reserve(per_type[t]); }
    }
    std::vector<std::pair<uint32_t, uint32_t>> world_range(F.worlds.size());
    for (size_t wi = 0; wi < F.worlds.size(); ++wi) {
        world_range[wi].first = (uint32_t)instances.size();
        for (InstBuild& ib : F.worlds[wi].inst) {
            if (ib.prims.empty()) continue;
            std::vector<BuildPrim> bp(ib.prims.size());
            parallel_chunks(ib.prims.size(), [&](size_t i_begin, size_t i_end) {
              for (size_t i = i_begin; i < i_end; ++i) {
                for (int a = 0; a < 3; ++a) { bp[i].bmin[a] = ib.prims[i].bmin[a]; bp[i].bmax[a] = ib.prims[i].bmax[a]; }
                bp[i].type = ib.prims[i].type;
                bp[i].src = (uint32_t)i;
                if (bp[i].type == PRIM_MOVING) {
                    // the SAH sees the sphere where it is in the middle of the shutter, not its union over the shutter: tall union
                    // boxes would keep static and moving spheres in the same subtrees, whose interpolated boxes are then tall too.
                    // The stored boxes (union in `nodes`, both shutter ends in `mnodes`) are refitted over the topology below.
                    const Node& mn = s->nodes[(size_t)ib.prims[i].node];
                    const double t0 = mn.d[6], t1 = mn.d[7], r = std::fabs(mn.d[8]), tm = 0.5 * (s->span0 + s->span1);
                    for (int a = 0; a < 3; ++a) {
                        const double c = mn.d[a] + ((tm - t0) / (t1 - t0)) * (mn.d[3 + a] - mn.d[a]);
                        bp[i].bmin[a] = c - r; bp[i].bmax[a] = c + r;
                    }
                }
              }
            });
            pt.lap("build prims");
            BuildResult br;
            bool built = false;
            if (allow_device_build && s->tuning.bvh_builder == 1 && bp.size() >= (size_t)std::max(16, s->tuning.bvh_device_min)) {
                // device LBVH (lbvh.cu): the host only rounds the boxes outward to f32 (+ pad), as BvhBuilder does for its nodes
                std::vector<float> fb(6 * bp.size());
                std::vector<uint8_t> ft(bp.size());
                for (size_t i = 0; i < bp.size(); ++i) {
                    for (int a = 0; a < 3; ++a) { fb[6 * i + a] = f32_floor(bp[i].bmin[a] - bo.pad); fb[6 * i + 3 + a] = f32_ceil(bp[i].bmax[a] + bo.pad); }
                    ft[i] = (uint8_t)bp[i].type;
                }
                if (nodes.size() & 1u) nodes.push_back(BvhNode32{});
                std::vector<BvhNode32> dn;
                float ms = 0.f;
                int depth = 0;
                const cudaError_t ce = lbvh_build_device(fb.data(), ft.data(), (uint32_t)bp.size(), (uint32_t)bo.max_leaf, (uint32_t)nodes.size(), cursor, dn,
                                                         br.leaf_order, &depth, &ms, &built);
                if (ce != cudaSuccess) return fail_cuda(ce, "device BVH build");
                if (built) {
                    br.root = (uint32_t)nodes.size();
                    br.max_depth = depth;
                    nodes.insert(nodes.end(), dn.begin(), dn.end());
                    HF.device_build_ms += ms;
                    HF.device_built_prims += (int64_t)bp.size();
                }
            }
            if (!built) {
                BvhBuilder builder(nodes, bo);
                br = builder.build(bp, cursor);
            }
            pt.lap(built ? "bvh build (device)" : "bvh build (host SAH)");
            if (built && pt.on) std::fprintf(stderr, "[rtb200 commit]   of which device kernels %8.3f ms (%zu primitives)\n", (double)HF.device_build_ms, bp.size());
            max_depth = std::max(max_depth, br.max_depth);
            // Triangles (the only mesh-sized type) are converted in parallel: slot k of this instance's triangles = the k-th triangle in
            // leaf order, so the arrays are those of the serial loop; every other type keeps the serial loop below.
            {
                const size_t n_lo = br.leaf_order.size();
                std::vector<uint32_t> tri_slot;
                size_t ntri = 0;
                for (size_t k = 0; k < n_lo; ++k) ntri += ib.prims[br.leaf_order[k]].type == PRIM_TRI ? 1u : 0u;
                if (ntri) {
                    tri_slot.resize(n_lo);
                    uint32_t c = 0;
                    for (size_t k = 0; k < n_lo; ++k) tri_slot[k] = ib.prims[br.leaf_order[k]].type == PRIM_TRI ? c++ : 0xffffffffu;
                    const size_t tri_base = tris.size(), meta_base = meta[PRIM_TRI].size(), mbox_base = mbox[PRIM_TRI].size();
                    tris.resize(tri_base + ntri);
                    meta[PRIM_TRI].resize(meta_base + ntri);
                    if (has_moving) mbox[PRIM_TRI].resize(mbox_base + ntri);
                    parallel_chunks(n_lo, [&](size_t k0, size_t k1) {
                        for (size_t k = k0; k < k1; ++k) {
                            if (tri_slot[k] == 0xffffffffu) continue;
                            const FlatPrim& p = ib.prims[br.leaf_order[k]];
                            const Node& n = s->nodes[(size_t)p.node];
                            if (has_moving) {
                                MotionBox mb;
                                for (int a = 0; a < 3; ++a) { mb.lo0[a] = mb.lo1[a] = p.bmin[a]; mb.hi0[a] = mb.hi1[a] = p.bmax[a]; }
                                mbox[PRIM_TRI][mbox_base + tri_slot[k]] = mb;
                            }
                            PrimMeta pm; pm.mat_id = p.mat; pm.prim_id = p.prim_id;
                            meta[PRIM_TRI][meta_base + tri_slot[k]] = pm;
                            const double *v0, *v1, *v2;
                            if (n.kind == N_MESH) {
                                const MeshData& m = *n.mesh;
                                v0 = &m.verts[3 * (size_t)m.faces[3 * (size_t)p.sub]];
                                v1 = &m.verts[3 * (size_t)m.faces[3 * (size_t)p.sub + 1]];
                                v2 = &m.verts[3 * (size_t)m.faces[3 * (size_t)p.sub + 2]];
                            } else {
                                v0 = &n.d[0]; v1 = &n.d[3]; v2 = &n.d[6];
                            }
                            // Triangle::new (hit.rs:96-107): unit normal of (v1-v0) x (v2-v0), computed in f64
                            const double ax = v1[0] - v0[0], ay = v1[1] - v0[1], az = v1[2] - v0[2];
                            const double bx = v2[0] - v0[0], by = v2[1] - v0[1], bz = v2[2] - v0[2];
                            double nx = ay * bz - az * by, ny = az * bx - ax * bz, nz = ax * by - ay * bx;
                            const double len = std::sqrt(nx * nx + ny * ny + nz * nz);
                            nx /= len; ny /= len; nz /= len;
                            DTri q;
                            for (int a = 0; a < 3; ++a) { q.v0[a] = (float)v0[a]; q.v1[a] = (float)v1[a]; q.v2[a] = (float)v2[a]; }
                            q.n[0] = (float)nx; q.n[1] = (float)ny; q.n[2] = (float)nz;
                            q.dd = -((double)q.n[0] * v0[0] + (double)q.n[1] * v0[1] + (double)q.n[2] * v0[2]); // rounded normal, exact vertex (rt_types.h)
                            q.pad_ = 0.0;
                            tris[tri_base + tri_slot[k]] = q;
                        }
                    });
                }
            }
            for (uint32_t src : br.leaf_order) {
                const FlatPrim& p = ib.prims[src];
                if (p.type == PRIM_TRI) continue; // done above
                const Node& n = s->nodes[(size_t)p.node];
                if (has_moving) { // box at the start and at the end of the shutter, in typed (leaf) order; static primitives: the same box twice
                    MotionBox mb;
                    for (int a = 0; a < 3; ++a) { mb.lo0[a] = mb.lo1[a] = p.bmin[a]; mb.hi0[a] = mb.hi1[a] = p.bmax[a]; }
                    if (p.type == PRIM_MOVING) {
                        const double t0 = n.d[6], t1 = n.d[7], r = n.d[8];
                        for (int a = 0; a < 3; ++a) {
                            const double c0 = n.d[a] + ((s->span0 - t0) / (t1 - t0)) * (n.d[3 + a] - n.d[a]);
                            const double c1 = n.d[a] + ((s->span1 - t0) / (t1 - t0)) * (n.d[3 + a] - n.d[a]);
                            mb.lo0[a] = c0 - std::fabs(r); mb.hi0[a] = c0 + std::fabs(r);
                            mb.lo1[a] = c1 - std::fabs(r); mb.hi1[a] = c1 + std::fabs(r);
                        }
                    }
                    mbox[p.type].push_back(mb);
                }
                PrimMeta pm; pm.mat_id = p.mat; pm.prim_id = p.prim_id;
                meta[p.type].push_back(pm);
                switch (p.type) {
                case PRIM_SPHERE: { DSphere q; q.cx = n.d[0]; q.cy = n.d[1]; q.cz = n.d[2]; q.r = n.d[3]; spheres.push_back(q); } break;
                case PRIM_MOVING: {
                    DMoving q;
                    for (int a = 0; a < 3; ++a) { q.c0[a] = n.d[a]; q.dc[a] = n.d[3 + a] - n.d[a]; }
                    q.t0 = n.d[6]; q.dt = n.d[7] - n.d[6]; q.r = n.d[8]; q.pad_ = 0;
                    movings.push_back(q);
                } break;
                case PRIM_GRAVITY: {
                    DGravity q;
                    int64_t i0, i1;
                    F.gravity_window(*n.grav, i0, i1);
                    q.x = n.d[0]; q.z = n.d[2]; q.r = n.d[4];
                    q.table_off = (int32_t)gtable.size(); q.idx0 = (int32_t)i0; q.n = (int32_t)(i1 - i0 + 1); q.pad_ = 0;
                    gtable.insert(gtable.end(), n.grav->begin() + i0, n.grav->begin() + i1 + 1);
                    gravities.push_back(q);
                } break;
                case PRIM_RECT: { DRect q; q.a0 = n.d[0]; q.a1 = n.d[1]; q.b0 = n.d[2]; q.b1 = n.d[3]; q.k = n.d[4]; q.axis = n.axis; q.pad_ = 0; rects.push_back(q); } break;
                case PRIM_BOX: { DBox q; for (int a = 0; a < 3; ++a) { q.p0[a] = n.d[a]; q.p1[a] = n.d[3 + a]; } boxes.push_back(q); } break;
                default: break;
                }
            }
            pt.lap("typed buffers");
            Instance in;
            in.root = br.root;
            in.chain_off = (uint32_t)ops.size();
            in.chain_len = (uint32_t)ib.chain.size();
            in.root4 = RT_WIDE_EMPTY;
            for (int a = 0; a < 3; ++a) { in.bmin[a] = nodes[br.root].min[a]; in.bmax[a] = nodes[br.root].max[a]; }
            ops.insert(ops.end(), ib.chain.begin(), ib.chain.end());
            instances.push_back(in);
        }
        world_range[wi].second = (uint32_t)instances.size();
    }
    if (max_depth > RT_BVH_MAX_DEPTH) return fail(RT_ERR_UNSUPPORTED, "BVH deeper than the traversal stack");
    if (!movings.empty()) { // motion-interpolated boxes: refit both shutter ends over the finished topology (post-order)
        HF.mnodes.assign(2 * nodes.size(), BvhNode32{});
        std::vector<MotionBox> nb(nodes.size());
        struct Item { uint32_t node; bool expanded; };
        for (const Instance& in : std::vector<Instance>(instances)) {
            std::vector<Item> st;
            st.push_back({in.root, false});
            while (!st.empty()) {
                Item it = st.back();
                st.pop_back();
                const BvhNode32& nd = nodes[it.node];
                MotionBox& b = nb[it.node];
                if (nd.count & RT_LEAF_FLAG) {
                    const uint32_t type = (nd.count >> 24) & 0x7fu, cnt = nd.count & 0xffffffu;
                    b.clear();
                    for (uint32_t k = 0; k < cnt; ++k) b.merge(mbox[type][nd.first + k]);
                } else if (!it.expanded) {
                    st.push_back({it.node, true});
                    st.push_back({nd.first, false});
                    st.push_back({nd.first + 1, false});
                    continue;
                } else {
                    b.clear();
                    b.merge(nb[nd.first]);
                    b.merge(nb[nd.first + 1]);
                }
                BvhNode32 m0 = nd, m1{};
                const bool empty = !(b.lo0[0] <= b.hi0[0]);
                for (int a = 0; a < 3; ++a) {
                    if (empty) { m0.min[a] = 3.0e38f; m0.max[a] = -3.0e38f; continue; } // the root pair's dummy sibling
                    m0.min[a] = f32_floor(b.lo0[a] - HF.pad); m0.max[a] = f32_ceil(b.hi0[a] + HF.pad);
                    const float lo1 = f32_floor(b.lo1[a] - HF.pad), hi1 = f32_ceil(b.hi1[a] + HF.pad);
                    m1.min[a] = f32_floor((double)lo1 - (double)m0.min[a]); // box0 + delta never pokes inside the box at the shutter's end
                    m1.max[a] = f32_ceil((double)hi1 - (double)m0.max[a]);
                }
                HF.mnodes[2 * (size_t)it.node] = m0;
                HF.mnodes[2 * (size_t)it.node + 1] = m1;
                if (!empty) { // `nodes`: the union over the shutter (MovingSphere::bounding_box, hit.rs:317-327) = union of the two end boxes
                    BvhNode32& un = nodes[it.node];
                    for (int a = 0; a < 3; ++a) {
                        un.min[a] = f32_floor(std::fmin(b.lo0[a], b.lo1[a]) - HF.pad);
                        un.max[a] = f32_ceil(std::fmax(b.hi0[a], b.hi1[a]) + HF.pad);
                    }
                }
            }
            // the root's sibling (empty leaf) keeps its inverted box
            HF.mnodes[2 * ((size_t)in.root + 1)] = nodes[in.root + 1];
        }
        for (Instance& in : instances)
            for (int a = 0; a < 3; ++a) { in.bmin[a] = nodes[in.root].min[a]; in.bmax[a] = nodes[in.root].max[a]; }
    }

    // materials: user materials first (ids = builder order), the phase functions of media were
    // appended to s->mats at rt_constant_medium time
    for (const MediumBuild& mb : F.media) {
        const Node& n = s->nodes[(size_t)mb.node];
        Medium m;
        m.inst_begin = world_range[mb.world].first;
        m.inst_end = world_range[mb.world].second;
        m.chain_off = (uint32_t)ops.size();
        m.chain_len = (uint32_t)mb.chain.size();
        ops.insert(ops.end(), mb.chain.begin(), mb.chain.end());
        m.mat_id = (uint32_t)n.mat;
        m.prim_id = (uint32_t)n.prim_base;
        m.neg_inv_density = -1.0 / n.d[0]; // hit.rs:949
        m.fast_type = 0; m.fast_idx = 0; m.fast_chain_off = 0; m.fast_chain_len = 0;
        if (m.inst_end - m.inst_begin == 1) {
            const Instance& bi = instances[m.inst_begin];
            const BvhNode32& rn = nodes[bi.root];
            const uint32_t lt = (rn.count >> 24) & 0x7fu, ln = rn.count & 0xffffffu;
            if ((rn.count & RT_LEAF_FLAG) && ln == 1 && (lt == PRIM_SPHERE || lt == PRIM_BOX)) {
                m.fast_type = lt == PRIM_SPHERE ? 1u : 2u;
                m.fast_idx = rn.first;
                m.fast_chain_off = bi.chain_off;
                m.fast_chain_len = bi.chain_len;
            }
        }
        media.push_back(m);
    }

    std::vector<DMaterial>& dmats = HF.dmats;
    dmats.resize(s->mats.size());
    for (size_t i = 0; i < s->mats.size(); ++i) {
        const MatDesc& m = s->mats[i];
        DMaterial d;
        std::memset(&d, 0, sizeof d);
        d.type = m.type;
        d.tex = (uint32_t)m.tex;
        d.flags = 0;
        if (m.type == MAT_LAMBERTIAN || m.type == MAT_LIGHT || m.type == MAT_ISOTROPIC) d.flags = tex_reads_uv(s, m.tex) ? 1u : 0u;
        for (int a = 0; a < 3; ++a) d.albedo[a] = (float)m.albedo[a];
        d.fuzz_or_ir = m.param;
        dmats[i] = d;
    }
    std::vector<DTexture>& dtex = HF.dtex;
    dtex.resize(s->tex.size());
    std::vector<PerlinTable>& perlin = HF.perlin;
    std::vector<float4>& texels = HF.texels;
    for (size_t i = 0; i < s->tex.size(); ++i) {
        const TexDesc& t = s->tex[i];
        DTexture d;
        std::memset(&d, 0, sizeof d);
        d.type = t.type;
        for (int a = 0; a < 3; ++a) d.rgb[a] = (float)t.rgb[a];
        if (t.type == TEX_CHECKER) { d.a = (uint32_t)t.a; d.b = (uint32_t)t.b; }
        else if (t.type == TEX_NOISE) { d.a = (uint32_t)perlin.size(); d.scale = t.scale; perlin.push_back(*t.perlin); }
        else if (t.type == TEX_IMAGE) {
            d.a = (uint32_t)texels.size(); d.w = (uint32_t)t.w; d.h = (uint32_t)t.h;
            const std::vector<float>& px = *t.texels;
            for (size_t k = 0; k + 3 < px.size() + 1; k += 4) texels.push_back(make_float4(px[k], px[k + 1], px[k + 2], px[k + 3]));
        }
        dtex[i] = d;
    }

    HF.n_main_instances = world_range[0].second - world_range[0].first;
    // 4-wide collapse of the main world's trees (boundary worlds of media keep the pair walk: their queries start at t_min = -inf).
    // Auto (measured on B200, tools/ab_wide.py): one wrapper-free instance without media that is plain spheres (book-1 final
    // +6 %) or a large triangle mesh (871 200 triangles +20 %); not GravitySphere scenes (-2 %).  rt_scene_set_bvh_width(4)
    // builds it for every main-world instance (the wavefront / generic kernels then walk it too: to be measured).
    const bool single_plain = HF.n_main_instances == 1 && media.empty() && instances[world_range[0].first].chain_len == 0;
    // (GravitySphere scenes, the animation config: -2 % on the wide tree in round 1, +11 % since the signed-row node test; MovingSphere
    // scenes, book-1 as shipped: -7.6 % with the min / max form of the motion nodes, +8.2 % with their signed rows:
    // profiles/r2_65_ab_wide_gravity_motion.txt, r2_66_ab_motion_signed.txt)
    const bool only_spheres = (!spheres.empty() || !movings.empty() || !gravities.empty()) && rects.empty() && boxes.empty() && tris.empty();
    const bool big_mesh = tris.size() >= 4096 && spheres.empty() && movings.empty() && gravities.empty() && boxes.empty();
    // round 2: the two primitive-mask-specialised media kernels of the wavefront (Cornell smoke, book-2 final: media with the
    // single-sphere / single-box fast path over spheres, moving spheres, rects and boxes) walk it too: +2.5 % / +3.4 % with the
    // signed-row node test (profiles/r2_59_ab_ext_wide.txt; it was +-0 with the min / max form)
    bool media_wave = !media.empty() && gravities.empty() && tris.empty();
    for (const Medium& m : media) media_wave = media_wave && m.fast_type != 0;
    if (HF.n_main_instances > 0 && (s->tuning.bvh_wide > 0 || (s->tuning.bvh_wide < 0 && ((single_plain && (only_spheres || big_mesh)) || media_wave)))) {
        bool all_ok = true;
        for (uint32_t i = world_range[0].first; i < world_range[0].second && all_ok; ++i) {
            const WideResult wr = collapse_to_wide(nodes, instances[i].root, HF.nodes4);
            all_ok = wr.ok;
            instances[i].root4 = wr.root;
            HF.wide_depth = std::max(HF.wide_depth, wr.max_depth);
        }
        if (!all_ok) { // a tree too deep or a leaf that does not fit a reference: the whole scene stays on sibling pairs
            HF.nodes4.clear();
            for (Instance& in : instances) in.root4 = RT_WIDE_EMPTY;
            HF.wide_depth = 0;
        }
        HF.root4 = instances[world_range[0].first].root4;
        if (!HF.nodes4.empty() && !HF.mnodes.empty()) build_motion_wide(HF.nodes4, HF.mnodes, HF.mnodes4);
        pt.lap("4-wide collapse");
    }
    return RT_OK;
}

// everything in DeviceScene that is not a pointer: counts, masks, kernel-selection flags, camera, background
void set_scene_scalars(const rt_scene* s, const HostFlat& HF, DeviceScene& D) {
    D.root4 = HF.root4;
    D.n_main_instances = HF.n_main_instances;
    D.n_media = (uint32_t)HF.media.size();
    D.n_prims = (uint32_t)s->n_prims;
    D.motion_t0 = s->span0;
    D.motion_inv_dt = s->span1 > s->span0 ? 1.0 / (s->span1 - s->span0) : 0.0;
    D.prim_mask = (HF.spheres.empty() ? 0u : 1u) | (HF.movings.empty() ? 0u : 2u) | (HF.gravities.empty() ? 0u : 4u) | (HF.rects.empty() ? 0u : 8u) |
                  (HF.boxes.empty() ? 0u : 16u) | (HF.tris.empty() ? 0u : 32u);
    D.flags = (!HF.rects.empty() || !HF.boxes.empty()) ? 1u : 0u;
    {
        bool all_fast = true;
        for (const Medium& m : HF.media) all_fast = all_fast && m.fast_type != 0;
        if (all_fast) D.flags |= 2u;
    }
    if (!HF.perlin.empty()) D.flags |= 8u;     // Perlin-noise textures: expensive, divergent shading
    if (!HF.texels.empty()) D.flags |= 16u;    // image textures (sphere uv needed)
    if (!HF.ops.empty()) D.flags |= 32u;       // Translate / RotateY wrappers present
    if (HF.tris.size() >= 4096) D.flags |= 4u; // deep triangle BVH: prefer the persistent warp-scheduled extend kernel
    if (s->camera.set) D.cam = s->camera.cam;
    for (int a = 0; a < 3; ++a) { D.background[a] = (float)s->background[a]; D.background_top[a] = (float)s->background_top[a]; }
    D.bg_gradient = s->bg_gradient ? 1u : 0u;
}

int32_t do_commit(rt_scene* s) {
    HostFlat HF;
    int dev_count = 0;
    cudaError_t ce = cudaGetDeviceCount(&dev_count);
    const bool have_device = ce == cudaSuccess && dev_count > 0;
    const int32_t fr = flatten_host(s, HF, have_device); // scene errors are reported before the missing device
    if (fr != RT_OK) return fr;
    if (!have_device) return fail(RT_ERR_CUDA, "no CUDA device: librtb200 has no CPU fallback");
    s->dev.device_built_prims = HF.device_built_prims;
    s->dev.device_build_ms = HF.device_build_ms;
    std::vector<BvhNode32>& nodes = HF.nodes;
    std::vector<DSphere>& spheres = HF.spheres; std::vector<DMoving>& movings = HF.movings; std::vector<DGravity>& gravities = HF.gravities;
    std::vector<double>& gtable = HF.gtable;
    std::vector<DRect>& rects = HF.rects; std::vector<DBox>& boxes = HF.boxes; std::vector<DTri>& tris = HF.tris;
    std::vector<PrimMeta>* meta = HF.meta;
    std::vector<Instance>& instances = HF.instances;
    std::vector<XformOp>& ops = HF.ops;
    std::vector<Medium>& media = HF.media;
    std::vector<DMaterial>& dmats = HF.dmats;
    std::vector<DTexture>& dtex = HF.dtex;
    std::vector<PerlinTable>& perlin = HF.perlin;
    std::vector<float4>& texels = HF.texels;

    s->dev.valid = false;
    DeviceScene& D = s->dev.scene;
    std::memset(&D, 0, sizeof D);
    UploadPlan up;
    up.add(nodes, D.nodes); up.add(HF.mnodes, D.mnodes); up.add(spheres, D.spheres); up.add(movings, D.movings); up.add(gravities, D.gravities); up.add(gtable, D.gravity_table);
    up.add(rects, D.rects); up.add(boxes, D.boxes); up.add(tris, D.tris);
    for (int t = 0; t < (int)PRIM_TYPE_COUNT; ++t) up.add(meta[t], D.meta[t]);
    up.add(instances, D.instances); up.add(ops, D.ops); up.add(media, D.media); up.add(dmats, D.materials); up.add(dtex, D.textures);
    up.add(perlin, D.perlin); up.add(texels, D.texels); up.add(HF.nodes4, D.nodes4); up.add(HF.mnodes4, D.mnodes4);
    if ((ce = up.run(s->dev)) != cudaSuccess) return fail_cuda(ce, "scene upload");
    if (HF.nodes4.empty()) D.nodes4 = nullptr;
    if (HF.mnodes4.empty()) D.mnodes4 = nullptr;
    if (HF.mnodes.empty()) D.mnodes = nullptr;
    set_scene_scalars(s, HF, D);
    cudaGetDevice(&s->dev.device);
    ++s->dev.generation;
    s->dev.valid = true;
    s->committed = true;
    return RT_OK;
}

} // namespace

extern "C" {

rt_scene* rt_scene_create(void) {
    rt_scene* s = new rt_scene();
    const char* e = std::getenv("RTB200_WAVE_SLOTS");
    if (e) s->tuning.wave_slots = (uint32_t)std::max(128L, std::atol(e));
    if ((e = std::getenv("RTB200_EXTEND_WAVES"))) s->tuning.extend_waves = std::atoi(e);
    if ((e = std::getenv("RTB200_MODE"))) s->tuning.mode = std::atoi(e);
    if ((e = std::getenv("RTB200_EXTEND_KIND"))) s->tuning.extend_kind = std::atoi(e);
    if ((e = std::getenv("RTB200_PRIM_SPECIALISE"))) s->tuning.prim_specialise = std::atoi(e);
    if ((e = std::getenv("RTB200_MEGA_WAIT"))) s->tuning.mega_wait = std::atoi(e);
    if ((e = std::getenv("RTB200_BVH_BUILDER"))) s->tuning.bvh_builder = (std::strcmp(e, "lbvh") == 0 || std::strcmp(e, "1") == 0) ? 1 : 0;
    if ((e = std::getenv("RTB200_BVH_DEVICE_MIN"))) s->tuning.bvh_device_min = std::atoi(e);
    if ((e = std::getenv("RTB200_BVH_WIDE"))) s->tuning.bvh_wide = std::atoi(e);
    return s;
}
void rt_scene_destroy(rt_scene* s) { delete s; }
const char* rt_last_error(void) { return g_err.c_str(); }
const char* rt_version(void) { return "rtb200 0.1 sm_100a (f64 rays / f32 slabs, wavefront)"; }

// ---------------------------------------------------------------- textures
int32_t rt_tex_solid(rt_scene* s, const double rgb[3]) {
    CHECK_SCENE(s);
    if (!rgb) return fail(RT_ERR_INVALID, "null colour");
    TexDesc t; t.type = TEX_SOLID;
    for (int a = 0; a < 3; ++a) t.rgb[a] = rgb[a];
    s->tex.push_back(t);
    return (int32_t)s->tex.size() - 1;
}
int32_t rt_tex_checker(rt_scene* s, int32_t even, int32_t odd) {
    CHECK_SCENE(s); CHECK_TEX(s, even); CHECK_TEX(s, odd);
    TexDesc t; t.type = TEX_CHECKER; t.a = even; t.b = odd;
    s->tex.push_back(t);
    return (int32_t)s->tex.size() - 1;
}
int32_t rt_tex_noise(rt_scene* s, double scale, const double* ranvec, const int32_t* px, const int32_t* py, const int32_t* pz, uint64_t seed) {
    CHECK_SCENE(s);
    PerlinTables gen;
    if (!ranvec || !px || !py || !pz) {
        perlin_generate(seed, gen);
        ranvec = gen.ranvec; px = gen.perm_x; py = gen.perm_y; pz = gen.perm_z;
    }
    auto pt = std::make_shared<PerlinTable>();
    for (int i = 0; i < 256; ++i) {
        for (int a = 0; a < 3; ++a) pt->ranvec[i][a] = ranvec[3 * i + a];
        if ((px[i] | py[i] | pz[i]) & ~255) return fail(RT_ERR_INVALID, "perm entry outside 0..255");
        pt->perm_x[i] = (uint8_t)px[i]; pt->perm_y[i] = (uint8_t)py[i]; pt->perm_z[i] = (uint8_t)pz[i];
    }
    TexDesc t; t.type = TEX_NOISE; t.scale = scale; t.perlin = pt;
    s->tex.push_back(t);
    return (int32_t)s->tex.size() - 1;
}
int32_t rt_tex_image(rt_scene* s, int32_t w, int32_t h, const double* rgb) {
    CHECK_SCENE(s);
    if (w <= 0 || h <= 0 || !rgb) return fail(RT_ERR_INVALID, "bad image");
    auto px = std::make_shared<std::vector<float>>((size_t)w * h * 4);
    for (size_t i = 0; i < (size_t)w * h; ++i) {
        (*px)[4 * i] = (float)rgb[3 * i]; (*px)[4 * i + 1] = (float)rgb[3 * i + 1]; (*px)[4 * i + 2] = (float)rgb[3 * i + 2]; (*px)[4 * i + 3] = 0.f;
    }
    TexDesc t; t.type = TEX_IMAGE; t.w = w; t.h = h; t.texels = px;
    s->tex.push_back(t);
    return (int32_t)s->tex.size() - 1;
}
int32_t rt_tex_image_ppm(rt_scene* s, const char* path) {
    CHECK_SCENE(s);
    if (!path) return fail(RT_ERR_INVALID, "null path");
    int32_t w, h;
    std::vector<double> rgb;
    std::string err;
    if (!read_ppm_any(path, w, h, rgb, err)) return fail(RT_ERR_IO, err); // P3 as the reference, or P6
    return rt_tex_image(s, w, h, rgb.data());
}

// ---------------------------------------------------------------- materials
static int32_t add_mat(rt_scene* s, const MatDesc& m) {
    s->mats.push_back(m);
    return (int32_t)s->mats.size() - 1;
}
int32_t rt_mat_lambertian(rt_scene* s, int32_t tex) { CHECK_SCENE(s); CHECK_TEX(s, tex); MatDesc m; m.type = MAT_LAMBERTIAN; m.tex = tex; return add_mat(s, m); }
int32_t rt_mat_metal(rt_scene* s, const double a[3], double fuzz) {
    CHECK_SCENE(s);
    if (!a) return fail(RT_ERR_INVALID, "null colour");
    MatDesc m; m.type = MAT_METAL;
    for (int i = 0; i < 3; ++i) m.albedo[i] = a[i];
    m.param = fuzz < 1.0 ? fuzz : 1.0; // hit.rs:1063
    return add_mat(s, m);
}
int32_t rt_mat_dielectric(rt_scene* s, double ir) { CHECK_SCENE(s); MatDesc m; m.type = MAT_DIELECTRIC; m.param = ir; return add_mat(s, m); }
int32_t rt_mat_diffuse_light(rt_scene* s, int32_t tex) { CHECK_SCENE(s); CHECK_TEX(s, tex); MatDesc m; m.type = MAT_LIGHT; m.tex = tex; return add_mat(s, m); }
int32_t rt_mat_isotropic(rt_scene* s, int32_t tex) { CHECK_SCENE(s); CHECK_TEX(s, tex); MatDesc m; m.type = MAT_ISOTROPIC; m.tex = tex; return add_mat(s, m); }

// ---------------------------------------------------------------- hittables
int32_t rt_sphere(rt_scene* s, const double c[3], double r, int32_t mat) {
    CHECK_SCENE(s); CHECK_MAT(s, mat);
    Node n; n.kind = N_SPHERE; n.mat = mat;
    n.d[0] = c[0]; n.d[1] = c[1]; n.d[2] = c[2]; n.d[3] = r;
    return add_node(s, std::move(n));
}
int32_t rt_moving_sphere(rt_scene* s, const double c0[3], const double c1[3], double t0, double t1, double r, int32_t mat) {
    CHECK_SCENE(s); CHECK_MAT(s, mat);
    if (!c0 || !c1) return fail(RT_ERR_INVALID, "null centre");
    if (!(t0 != t1)) return fail(RT_ERR_INVALID, "MovingSphere with time0 == time1: get_center divides by zero (hit.rs:275-278)");
    Node n; n.kind = N_MOVING; n.mat = mat;
    for (int a = 0; a < 3; ++a) { n.d[a] = c0[a]; n.d[3 + a] = c1[a]; }
    n.d[6] = t0; n.d[7] = t1; n.d[8] = r;
    return add_node(s, std::move(n));
}
int32_t rt_gravity_sphere(rt_scene* s, const double st[3], double time0, double r, int32_t mat) {
    CHECK_SCENE(s); CHECK_MAT(s, mat);
    Node n; n.kind = N_GRAVITY; n.mat = mat;
    n.d[0] = st[0]; n.d[1] = st[1]; n.d[2] = st[2]; n.d[3] = time0; n.d[4] = r;
    // GravitySphere::new (hit.rs:346-359): explicit Euler bounce table, one entry per 0.001 of time up to 100
    auto tab = std::make_shared<std::vector<double>>();
    tab->reserve(100002);
    tab->push_back(st[1]);
    const double incr = 0.001;
    double t = time0, y = st[1], vel = 0.0;
    while (t < 100.0) {
        t += incr;
        vel -= 0.000001;
        if (y - 1.0 * r <= 0.0) vel *= -0.92;
        y = std::fmax(1.0 * r, y + vel);
        tab->push_back(y);
    }
    n.grav = tab;
    return add_node(s, std::move(n));
}
static int32_t add_rect(rt_scene* s, int axis, double a0, double a1, double b0, double b1, double k, int32_t mat) {
    Node n; n.kind = N_RECT; n.mat = mat; n.axis = axis;
    n.d[0] = a0; n.d[1] = a1; n.d[2] = b0; n.d[3] = b1; n.d[4] = k;
    return add_node(s, std::move(n));
}
int32_t rt_xy_rect(rt_scene* s, double x0, double x1, double y0, double y1, double k, int32_t mat) { CHECK_SCENE(s); CHECK_MAT(s, mat); return add_rect(s, 2, x0, x1, y0, y1, k, mat); }
int32_t rt_xz_rect(rt_scene* s, double x0, double x1, double z0, double z1, double k, int32_t mat) { CHECK_SCENE(s); CHECK_MAT(s, mat); return add_rect(s, 1, x0, x1, z0, z1, k, mat); }
int32_t rt_yz_rect(rt_scene* s, double y0, double y1, double z0, double z1, double k, int32_t mat) { CHECK_SCENE(s); CHECK_MAT(s, mat); return add_rect(s, 0, y0, y1, z0, z1, k, mat); }
int32_t rt_box(rt_scene* s, const double p0[3], const double p1[3], int32_t mat) {
    CHECK_SCENE(s); CHECK_MAT(s, mat);
    Node n; n.kind = N_BOX; n.mat = mat;
    for (int a = 0; a < 3; ++a) { n.d[a] = p0[a]; n.d[3 + a] = p1[a]; }
    return add_node(s, std::move(n));
}
int32_t rt_triangle(rt_scene* s, const double v0[3], const double v1[3], const double v2[3], int32_t mat) {
    CHECK_SCENE(s); CHECK_MAT(s, mat);
    Node n; n.kind = N_TRI; n.mat = mat;
    for (int a = 0; a < 3; ++a) { n.d[a] = v0[a]; n.d[3 + a] = v1[a]; n.d[6 + a] = v2[a]; }
    return add_node(s, std::move(n));
}
int32_t rt_triangle_mesh(rt_scene* s, const double* verts, int64_t nv, const uint32_t* idx, int64_t nt, int32_t mat) {
    CHECK_SCENE(s); CHECK_MAT(s, mat);
    if (!verts || !idx || nv <= 0 || nt < 0) return fail(RT_ERR_INVALID, "bad mesh");
    for (int64_t i = 0; i < 3 * nt; ++i)
        if (idx[i] >= (uint64_t)nv) return fail(RT_ERR_INVALID, "mesh index out of range");
    Node n; n.kind = N_MESH; n.mat = mat;
    n.mesh = std::make_shared<MeshData>();
    n.mesh->verts.assign(verts, verts + 3 * nv);
    n.mesh->faces.assign(idx, idx + 3 * nt);
    return add_node(s, std::move(n));
}
int32_t rt_ply_load(rt_scene* s, const char* path, double scale, int32_t mat) {
    CHECK_SCENE(s); CHECK_MAT(s, mat);
    if (!path) return fail(RT_ERR_INVALID, "null path");
    Node n; n.kind = N_MESH; n.mat = mat;
    n.mesh = std::make_shared<MeshData>();
    std::string err;
    if (!read_ply_any(path, scale, n.mesh->verts, n.mesh->faces, err)) return fail(RT_ERR_IO, err); // ASCII as the reference, or binary_little_endian
    return add_node(s, std::move(n));
}
int32_t rt_list(rt_scene* s, const int32_t* ids, int32_t cnt) {
    CHECK_SCENE(s);
    if (cnt < 0 || (cnt > 0 && !ids)) return fail(RT_ERR_INVALID, "bad list");
    Node n; n.kind = N_LIST;
    for (int32_t i = 0; i < cnt; ++i) { CHECK_OBJ(s, ids[i]); n.children.push_back(ids[i]); }
    return add_node(s, std::move(n));
}
int32_t rt_bvh(rt_scene* s, const int32_t* ids, int32_t cnt, double t0, double t1) {
    CHECK_SCENE(s);
    if (cnt < 0 || (cnt > 0 && !ids)) return fail(RT_ERR_INVALID, "bad list");
    Node n; n.kind = N_BVH; n.d[0] = t0; n.d[1] = t1;
    for (int32_t i = 0; i < cnt; ++i) { CHECK_OBJ(s, ids[i]); n.children.push_back(ids[i]); }
    // BvhNode::new unwraps bounding boxes (bvh.rs:27-28): an empty group panics in the reference
    bool empty = n.children.empty();
    if (cnt == 1) {
        const Node& c = s->nodes[(size_t)ids[0]];
        if ((c.kind == N_LIST && c.children.empty()) || (c.kind == N_MESH && c.mesh->faces.empty())) empty = true;
    }
    if (empty) return fail(RT_ERR_EMPTY, "BvhNode over an empty list (the reference panics, bvh.rs:27-28)");
    return add_node(s, std::move(n));
}
int32_t rt_translate(rt_scene* s, const double off[3], int32_t child) {
    CHECK_SCENE(s); CHECK_OBJ(s, child);
    Node n; n.kind = N_TRANSLATE; n.d[0] = off[0]; n.d[1] = off[1]; n.d[2] = off[2];
    n.children.push_back(child);
    return add_node(s, std::move(n));
}
int32_t rt_rotate_y(rt_scene* s, double angle_deg, int32_t child) {
    CHECK_SCENE(s); CHECK_OBJ(s, child);
    Node n; n.kind = N_ROTY;
    const double angle = angle_deg * (3.14159265358979323846264338327950288 / 180.0); // f64::to_radians (hit.rs:844)
    n.d[0] = std::sin(angle); n.d[1] = std::cos(angle);
    n.children.push_back(child);
    return add_node(s, std::move(n));
}
int32_t rt_constant_medium(rt_scene* s, const double rgb[3], double density, int32_t boundary) {
    CHECK_SCENE(s); CHECK_OBJ(s, boundary);
    // ConstantMedium::from_color builds its own Isotropic(SolidColor(c)) (hit.rs:945-951): it takes
    // the next texture and material ids
    const int32_t tex = rt_tex_solid(s, rgb);
    if (tex < 0) return tex;
    const int32_t mat = rt_mat_isotropic(s, tex);
    Node n; n.kind = N_MEDIUM; n.mat = mat; n.d[0] = density;
    n.children.push_back(boundary);
    return add_node(s, std::move(n));
}

// ---------------------------------------------------------------- scene
int32_t rt_scene_set_root(rt_scene* s, int32_t id) {
    CHECK_SCENE(s); CHECK_OBJ(s, id);
    s->root = id;
    s->committed = false;
    return RT_OK;
}
int32_t rt_scene_set_camera_fields(rt_scene* s, const double f[24]) {
    CHECK_SCENE(s);
    if (!f) return fail(RT_ERR_INVALID, "null camera fields");
    DCamera& c = s->camera.cam;
    for (int a = 0; a < 3; ++a) {
        c.origin[a] = f[a]; c.lower_left_corner[a] = f[3 + a]; c.horizontal[a] = f[6 + a]; c.vertical[a] = f[9 + a];
        c.u[a] = f[12 + a]; c.v[a] = f[15 + a]; c.w[a] = f[18 + a];
    }
    c.lens_radius = f[21]; c.time1 = f[22]; c.time2 = f[23];
    s->camera.set = true;
    s->committed = false; // moving-primitive bounds depend on the shutter
    return RT_OK;
}
int32_t rt_scene_set_camera(rt_scene* s, const double lf[3], const double la[3], const double vup[3], double vfov, double aspect, double aperture,
                            double focus_dist, double t1, double t2) {
    CHECK_SCENE(s);
    if (!lf || !la || !vup) return fail(RT_ERR_INVALID, "null camera vector");
    // Camera::new (camera.rs:20-57)
    const double theta = vfov * (3.14159265358979323846264338327950288 / 180.0);
    const double h = std::tan(theta / 2.0);
    const double viewport_height = 2.0 * h;
    const double viewport_width = aspect * viewport_height;
    double w[3] = {lf[0] - la[0], lf[1] - la[1], lf[2] - la[2]};
    const double wl = std::sqrt(w[0] * w[0] + w[1] * w[1] + w[2] * w[2]);
    for (int a = 0; a < 3; ++a) w[a] /= wl;
    double u[3] = {vup[1] * w[2] - vup[2] * w[1], vup[2] * w[0] - vup[0] * w[2], vup[0] * w[1] - vup[1] * w[0]};
    const double ul = std::sqrt(u[0] * u[0] + u[1] * u[1] + u[2] * u[2]);
    for (int a = 0; a < 3; ++a) u[a] /= ul;
    const double v[3] = {w[1] * u[2] - w[2] * u[1], w[2] * u[0] - w[0] * u[2], w[0] * u[1] - w[1] * u[0]};
    DCamera& c = s->camera.cam;
    for (int a = 0; a < 3; ++a) {
        c.origin[a] = lf[a];
        c.u[a] = u[a]; c.v[a] = v[a]; c.w[a] = w[a];
        c.horizontal[a] = focus_dist * viewport_width * u[a];
        c.vertical[a] = focus_dist * viewport_height * v[a];
    }
    for (int a = 0; a < 3; ++a) c.lower_left_corner[a] = c.origin[a] - c.horizontal[a] / 2.0 - c.vertical[a] / 2.0 - focus_dist * w[a];
    c.lens_radius = aperture / 2.0;
    c.time1 = t1; c.time2 = t2;
    s->camera.set = true;
    s->committed = false; // moving-primitive bounds depend on the shutter
    return RT_OK;
}
int32_t rt_scene_set_background(rt_scene* s, const double rgb[3]) {
    CHECK_SCENE(s);
    if (!rgb) return fail(RT_ERR_INVALID, "null colour");
    for (int a = 0; a < 3; ++a) s->background[a] = rgb[a];
    s->bg_gradient = false;
    if (s->dev.valid) {
        for (int a = 0; a < 3; ++a) s->dev.scene.background[a] = (float)rgb[a];
        s->dev.scene.bg_gradient = 0u;
    }
    return RT_OK;
}
int32_t rt_scene_set_background_gradient(rt_scene* s, const double horizon[3], const double zenith[3]) {
    CHECK_SCENE(s);
    if (!horizon || !zenith) return fail(RT_ERR_INVALID, "null colour");
    for (int a = 0; a < 3; ++a) { s->background[a] = horizon[a]; s->background_top[a] = zenith[a]; }
    s->bg_gradient = true;
    if (s->dev.valid) {
        for (int a = 0; a < 3; ++a) { s->dev.scene.background[a] = (float)horizon[a]; s->dev.scene.background_top[a] = (float)zenith[a]; }
        s->dev.scene.bg_gradient = 1u;
    }
    return RT_OK;
}
int32_t rt_scene_commit(rt_scene* s) {
    CHECK_SCENE(s);
    return do_commit(s);
}
int32_t rt_world_build(rt_scene* s, int32_t scene_id, uint64_t seed, int32_t param) {
    CHECK_SCENE(s);
    return build_world(s, scene_id, seed, param);
}
int32_t rt_scene_num_prims(rt_scene* s) {
    CHECK_SCENE(s);
    return s->n_prims;
}

// ---------------------------------------------------------------- render
int32_t rt_image_height(const rt_render_config* cfg) {
    if (!cfg || cfg->image_width <= 0 || !(cfg->aspect_ratio > 0)) return RT_ERR_INVALID;
    const double h = (double)cfg->image_width / cfg->aspect_ratio; // world.rs:1192, `as i32` saturates
    if (h != h) return 0;
    if (h >= 2147483647.0) return 2147483647;
    return (int32_t)h;
}

static int32_t make_job(rt_scene* s, const rt_render_config* cfg, RenderJob& job) {
    if (!cfg) return fail(RT_ERR_INVALID, "null config");
    if (!s->committed || !s->dev.valid) return fail(RT_ERR_STATE, "scene not committed");
    if (!s->camera.set) return fail(RT_ERR_STATE, "no camera");
    if (cfg->image_width <= 0 || cfg->samples_per_pixel <= 0 || cfg->max_depth <= 0) return fail(RT_ERR_INVALID, "Config::new assert (world.rs:36-40)");
    const int32_t H = rt_image_height(cfg);
    if (H <= 0) return fail(RT_ERR_INVALID, "image height <= 0 (Screen::new assert, screen.rs:14)");
    if ((int64_t)cfg->image_width * H > (int64_t)1 << 30) return fail(RT_ERR_INVALID, "image too large");
    job.width = cfg->image_width;
    job.height = H;
    job.rows = cfg->compat_threads > 0 ? (H / cfg->compat_threads) * cfg->compat_threads : H; // world.rs:1198-1202
    job.spp_total = cfg->samples_per_pixel;
    job.sample_begin = cfg->sample_begin;
    job.sample_end = cfg->sample_end == 0 ? cfg->samples_per_pixel : cfg->sample_end;
    if (job.sample_begin < 0 || job.sample_end > job.spp_total || job.sample_begin > job.sample_end) return fail(RT_ERR_INVALID, "bad sample range");
    job.max_depth = cfg->max_depth;
    job.seed = cfg->seed;
    job.tile_count = RT_RENDER_TILE_COUNT(cfg->flags) > 1 ? RT_RENDER_TILE_COUNT(cfg->flags) : 1;
    job.tile_rank = job.tile_count > 1 ? RT_RENDER_TILE_RANK(cfg->flags) : 0;
    if (job.tile_rank >= job.tile_count) return fail(RT_ERR_INVALID, "tile shard rank >= count");
    return RT_OK;
}

static RenderTuning tuning_for_flags(const rt_scene* s, const rt_render_config* cfg) {
    RenderTuning tune = s->tuning;
    tune.timed_extend = (cfg->flags & RT_RENDER_TIMED_EXTEND) ? 1 : 0;
    tune.count_events = (cfg->flags & RT_RENDER_COUNT_EVENTS) ? 1 : 0;
    if (cfg->flags & RT_RENDER_FORCE_WAVEFRONT) tune.mode = RT_MODE_WAVEFRONT;
    if (cfg->flags & RT_RENDER_FORCE_FUSED) tune.mode = RT_MODE_FUSED;
    if (cfg->flags & RT_RENDER_FORCE_POOL) tune.mode = RT_MODE_POOL;
    if (tune.timed_extend || tune.count_events) tune.mode = RT_MODE_WAVEFRONT; // both are diagnostics of the wavefront's k_extend
    return tune;
}

int32_t rt_render_device(rt_scene* s, const rt_render_config* cfg, int64_t* d_accum, void* cuda_stream, rt_stats* stats) {
    CHECK_SCENE(s);
    if (!d_accum) return fail(RT_ERR_INVALID, "null accumulator");
    RenderJob job;
    const int32_t r = make_job(s, cfg, job);
    if (r != RT_OK) return r;
    if (stats) std::memset(stats, 0, sizeof *stats);
    const auto t0 = std::chrono::steady_clock::now();
    RenderTuning tune = tuning_for_flags(s, cfg);
    tune.no_wait = (cfg->flags & RT_RENDER_NO_WAIT) ? 1 : 0;
    const cudaError_t e = launch_render(s->dev.scene, job, tune, d_accum, (cudaStream_t)cuda_stream, stats, &s->workspace);
    if (e != cudaSuccess) return fail_cuda(e, "render");
    if (stats) stats->ms_total = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    return RT_OK;
}

int32_t rt_render_device_paths(rt_scene* s, const rt_render_config* cfg, uint64_t path_begin, uint64_t path_end, int64_t* d_accum, void* cuda_stream, rt_stats* stats) {
    CHECK_SCENE(s);
    if (!d_accum) return fail(RT_ERR_INVALID, "null accumulator");
    RenderJob job;
    const int32_t r = make_job(s, cfg, job);
    if (r != RT_OK) return r;
    if (path_begin > path_end) return fail(RT_ERR_INVALID, "bad path range");
    if (path_begin == path_end) { // an empty shard renders nothing
        if (stats) std::memset(stats, 0, sizeof *stats);
        return RT_OK;
    }
    job.path_begin = path_begin; job.path_end = path_end;
    if (stats) std::memset(stats, 0, sizeof *stats);
    const auto t0 = std::chrono::steady_clock::now();
    RenderTuning tune = tuning_for_flags(s, cfg);
    tune.no_wait = (cfg->flags & RT_RENDER_NO_WAIT) ? 1 : 0;
    const cudaError_t e = launch_render(s->dev.scene, job, tune, d_accum, (cudaStream_t)cuda_stream, stats, &s->workspace);
    if (e != cudaSuccess) return fail_cuda(e, "render");
    if (stats) stats->ms_total = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    return RT_OK;
}

int32_t rt_resolve_device(const int64_t* d_accum, double* d_screen, int32_t width, int32_t height, int32_t spp, int32_t rendered_rows, void* cuda_stream) {
    if (!d_accum || !d_screen || width <= 0 || height <= 0 || spp <= 0) return fail(RT_ERR_INVALID, "bad resolve arguments");
    const cudaError_t e = launch_resolve(d_accum, d_screen, width, height, spp, rendered_rows, (cudaStream_t)cuda_stream);
    if (e != cudaSuccess) return fail_cuda(e, "resolve");
    return RT_OK;
}

// ---- rt_render / rt_render_multi: host-buffer entry points (what a Rust render_scene_gpu calls, world.rs:1181-1247)
namespace {

// The host-buffer entry points run on the device the scene was committed on, whatever device is current in the calling thread, and
// leave the caller's current device as they found it.
struct DeviceGuard {
    int home = -1;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&home) != cudaSuccess) home = -1;
        if (home != dev) cudaSetDevice(dev);
    }
    ~DeviceGuard() {
        int cur = -1;
        if (home >= 0 && cudaGetDevice(&cur) == cudaSuccess && cur != home) cudaSetDevice(home);
    }
};

int32_t ensure_out_buffers(rt_scene* s, size_t n) {
    RenderBuffers& o = s->out;
    cudaError_t e;
    if (!o.stream && (e = cudaStreamCreateWithFlags(&o.stream, cudaStreamNonBlocking)) != cudaSuccess) return fail_cuda(e, "stream");
    if (n <= o.cap) return RT_OK;
    cudaStream_t keep = o.stream;
    o.stream = nullptr;
    o.release();
    o.stream = keep;
    if ((e = cudaMalloc(&o.d_accum, n * sizeof(int64_t))) != cudaSuccess) return fail_cuda(e, "accumulator allocation");
    if ((e = cudaMalloc(&o.d_u8, n)) != cudaSuccess) return fail_cuda(e, "screen allocation");
    if ((e = cudaMallocHost(&o.h_u8, n)) != cudaSuccess) return fail_cuda(e, "pinned screen allocation");
    o.cap = n;
    return RT_OK;
}

// Screen bytes (every value is an integer 0..255, vec3.rs:89-107) -> the reference's f64 Colors
void widen_screen(const uint8_t* src, double* dst, size_t n) {
    for (size_t i = 0; i < n; ++i) dst[i] = (double)src[i];
}

// sum of the shards (own + peers) -> out buffers on the gathering GPU -> host
int32_t gather_and_copy_out(rt_scene* s, const AccumShards& shards, const RenderJob& job, double* out_screen, int64_t* out_accum) {
    RenderBuffers& o = s->out;
    const size_t n = (size_t)job.width * job.height * 3;
    cudaError_t e;
    // one shard: its sums already are o.d_accum; several: summed in place over shard 0 (a thread reads element i of every shard before it writes it)
    int64_t* sum_out = (out_accum && shards.n > 1) ? o.d_accum : nullptr;
    if ((e = launch_reduce_resolve(shards, sum_out, out_screen ? o.d_u8 : nullptr, nullptr, job.width, job.height, job.spp_total, job.rows, o.stream)) != cudaSuccess)
        return fail_cuda(e, "reduce + resolve");
    if (out_screen && (e = cudaMemcpyAsync(o.h_u8, o.d_u8, n, cudaMemcpyDeviceToHost, o.stream)) != cudaSuccess) return fail_cuda(e, "screen copy");
    if (out_accum && (e = cudaMemcpyAsync(out_accum, o.d_accum, n * sizeof(int64_t), cudaMemcpyDeviceToHost, o.stream)) != cudaSuccess) return fail_cuda(e, "accum copy");
    if ((e = cudaStreamSynchronize(o.stream)) != cudaSuccess) return fail_cuda(e, "render sync");
    if (out_screen) widen_screen(o.h_u8, out_screen, n);
    return RT_OK;
}

RenderTuning tuning_for(const rt_scene* s, const rt_render_config* cfg) { return tuning_for_flags(s, cfg); }

} // namespace

int32_t rt_render(rt_scene* s, const rt_render_config* cfg, double* out_screen, int64_t* out_accum, rt_stats* stats) {
    CHECK_SCENE(s);
    RenderJob job;
    int32_t rc = make_job(s, cfg, job);
    if (rc != RT_OK) return rc;
    const auto t0 = std::chrono::steady_clock::now();
    DeviceGuard guard(s->dev.device);
    const size_t n = (size_t)job.width * job.height * 3;
    if ((rc = ensure_out_buffers(s, n)) != RT_OK) return rc;
    RenderBuffers& o = s->out;
    cudaError_t e;
    if ((e = cudaMemsetAsync(o.d_accum, 0, n * sizeof(int64_t), o.stream)) != cudaSuccess) return fail_cuda(e, "memset");
    if (stats) std::memset(stats, 0, sizeof *stats);
    if ((e = launch_render(s->dev.scene, job, tuning_for(s, cfg), o.d_accum, o.stream, stats, &s->workspace)) != cudaSuccess) return fail_cuda(e, "render");
    AccumShards sh;
    std::memset(&sh, 0, sizeof sh);
    sh.n = 1;
    sh.p[0] = o.d_accum;
    if ((rc = gather_and_copy_out(s, sh, job, out_screen, out_accum)) != RT_OK) return rc;
    if (stats) stats->ms_total = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    return RT_OK;
}

// ---- adaptive sampling (include/rtb200.h rt_render_adaptive; the numpy mirror is ray_tracing_series_rust_b200/adaptive.py)
namespace {

int32_t ensure_adaptive_buffers(rt_scene* s, size_t npix) {
    AdaptiveBuffers& b = s->adaptive;
    if (npix <= b.cap) return RT_OK;
    b.release();
    cudaError_t e;
    const size_t temp = adaptive_select_temp_bytes((uint32_t)npix);
    if ((e = cudaMalloc(&b.d_a, npix * 3 * sizeof(int64_t))) != cudaSuccess || (e = cudaMalloc(&b.d_b, npix * 3 * sizeof(int64_t))) != cudaSuccess ||
        (e = cudaMalloc(&b.d_list[0], npix * sizeof(uint32_t))) != cudaSuccess || (e = cudaMalloc(&b.d_list[1], npix * sizeof(uint32_t))) != cudaSuccess ||
        (e = cudaMalloc(&b.d_samples, npix * sizeof(int32_t))) != cudaSuccess || (e = cudaMalloc(&b.d_u, npix)) != cudaSuccess ||
        (e = cudaMalloc(&b.d_keep, npix)) != cudaSuccess || (e = cudaMalloc(&b.d_temp, std::max<size_t>(temp, 1))) != cudaSuccess ||
        (e = cudaMallocHost(&b.h_count, sizeof(uint32_t))) != cudaSuccess) {
        b.release();
        return fail_cuda(e, "adaptive buffers");
    }
    b.temp_bytes = temp;
    b.cap = npix;
    return RT_OK;
}

// Counters of several renders into one rt_stats.  concurrent: the renders ran at the same time (rt_render_multi's shards), so
// iterations and device times are those of the slowest; otherwise (rt_render_adaptive's rounds, one after the other) they add up.
void add_stats(rt_stats& sum, const rt_stats& r, bool concurrent) {
    sum.paths += r.paths;
    sum.segments += r.segments;
    sum.box_tests += r.box_tests;
    for (int i = 0; i < 8; ++i) sum.prim_tests[i] += r.prim_tests[i];
    for (int i = 0; i < 5; ++i) sum.scatters[i] += r.scatters[i];
    sum.medium_queries += r.medium_queries;
    sum.kernel_launches += r.kernel_launches;
    if (concurrent) {
        sum.iterations = std::max(sum.iterations, r.iterations);
        sum.ms_device = std::max(sum.ms_device, r.ms_device);
        sum.ms_extend = std::max(sum.ms_extend, r.ms_extend);
    } else {
        sum.iterations += r.iterations;
        sum.ms_device += r.ms_device;
        sum.ms_extend += r.ms_extend;
    }
}

} // namespace

// ---- multi-GPU inside the library (SURVEY.md 8(b) n_gpus / shard_mode, 8(e)): one process, N devices
namespace {

bool multi_alias() { // test hook: every logical GPU is the scene's own device (separate arenas, accumulators and streams): 1-GPU boxes run the N-GPU logic
    const char* e = std::getenv("RTB200_MULTI_ALIAS");
    return e && std::atoi(e) != 0;
}

// logical GPU g (>= 1) -> physical device: the devices after the scene's own, wrapping around
int32_t replica_device(const rt_scene* s, int g, int dev_count) { return multi_alias() ? s->dev.device : (s->dev.device + g) % dev_count; }

int32_t ensure_replicas(rt_scene* s, int32_t n_gpus, size_t accum_elems) {
    int dev_count = 0;
    cudaError_t e = cudaGetDeviceCount(&dev_count);
    if (e != cudaSuccess || dev_count < 1) return fail(RT_ERR_CUDA, "no CUDA device: librtb200 has no CPU fallback");
    if (n_gpus > RT_MAX_GPUS) return fail(RT_ERR_INVALID, "n_gpus > 16");
    if (n_gpus > dev_count && !multi_alias()) return fail(RT_ERR_INVALID, "n_gpus exceeds the visible CUDA devices");
    if ((int)s->replicas.size() < n_gpus - 1) s->replicas.resize((size_t)n_gpus - 1);
    int home = 0;
    cudaGetDevice(&home);
    int32_t rc = RT_OK;
    for (int g = 1; g < n_gpus && rc == RT_OK; ++g) {
        Replica& r = s->replicas[(size_t)g - 1];
        const int dev = replica_device(s, g, dev_count);
        if (r.device != dev) { r.release(); r = Replica(); r.device = dev; }
        if ((e = cudaSetDevice(dev)) != cudaSuccess) { rc = fail_cuda(e, "cudaSetDevice"); break; }
        if (!r.stream && (e = cudaStreamCreateWithFlags(&r.stream, cudaStreamNonBlocking)) != cudaSuccess) { rc = fail_cuda(e, "replica stream"); break; }
        if (r.generation != s->dev.generation) { // upload the committed bytes (still in the pinned staging buffer) to this GPU
            if (s->dev.bytes > r.capacity) {
                if (r.arena) cudaFree(r.arena);
                r.arena = nullptr; r.capacity = 0;
                const size_t cap = s->dev.bytes + s->dev.bytes / 4 + 4096;
                if ((e = cudaMalloc(&r.arena, cap)) != cudaSuccess) { rc = fail_cuda(e, "replica arena"); break; }
                r.capacity = cap;
            }
            if ((e = cudaMemcpyAsync(r.arena, s->dev.staging, s->dev.bytes, cudaMemcpyHostToDevice, r.stream)) != cudaSuccess) { rc = fail_cuda(e, "replica upload"); break; }
            r.generation = s->dev.generation;
        }
        if (accum_elems > r.accum_cap) {
            if (r.d_accum) cudaFree(r.d_accum);
            r.d_accum = nullptr; r.accum_cap = 0;
            if ((e = cudaMalloc(&r.d_accum, accum_elems * sizeof(int64_t))) != cudaSuccess) { rc = fail_cuda(e, "replica accumulator"); break; }
            r.accum_cap = accum_elems;
        }
        // scalars (camera, background, flags) follow the primary scene; pointers are re-based into this arena
        r.scene = s->dev.scene;
        for (const auto& fo : s->dev.layout) {
            const char** field = reinterpret_cast<const char**>(reinterpret_cast<char*>(&r.scene) + fo.first);
            if (*field) *field = r.arena + fo.second;
        }
        // peer access: the gathering GPU (the scene's own) reads this accumulator in k_reduce_resolve
        r.peer_ok = dev == s->dev.device;
        if (!r.peer_ok) {
            int can = 0;
            cudaDeviceCanAccessPeer(&can, s->dev.device, dev);
            if (can) {
                cudaSetDevice(s->dev.device);
                e = cudaDeviceEnablePeerAccess(dev, 0);
                if (e == cudaSuccess || e == cudaErrorPeerAccessAlreadyEnabled) r.peer_ok = true;
                (void)cudaGetLastError();
            }
            if (!r.peer_ok && accum_elems > r.stage_cap) { // no P2P route: the shard is copied next to the gathering GPU's own first
                cudaSetDevice(s->dev.device);
                if (r.d_stage) cudaFree(r.d_stage);
                r.d_stage = nullptr; r.stage_cap = 0;
                if ((e = cudaMalloc(&r.d_stage, accum_elems * sizeof(int64_t))) != cudaSuccess) { rc = fail_cuda(e, "gather staging"); break; }
                r.stage_cap = accum_elems;
            }
        }
    }
    cudaSetDevice(home);
    return rc;
}

} // namespace

int32_t rt_scene_commit_multi(rt_scene* s, int32_t n_gpus) {
    CHECK_SCENE(s);
    if (n_gpus < 1) return fail(RT_ERR_INVALID, "n_gpus < 1");
    const int32_t rc = do_commit(s);
    if (rc != RT_OK) return rc;
    return ensure_replicas(s, n_gpus, 0);
}

int32_t rt_render_multi(rt_scene* s, const rt_render_config* cfg, int32_t n_gpus, int32_t shard_mode, double* out_screen, int64_t* out_accum, rt_stats* stats) {
    CHECK_SCENE(s);
    if (n_gpus < 1) return fail(RT_ERR_INVALID, "n_gpus < 1");
    if (shard_mode != RT_SHARD_SAMPLES && shard_mode != RT_SHARD_TILES) return fail(RT_ERR_INVALID, "shard_mode must be RT_SHARD_SAMPLES or RT_SHARD_TILES");
    if (n_gpus == 1) return rt_render(s, cfg, out_screen, out_accum, stats);
    RenderJob job;
    int32_t rc = make_job(s, cfg, job);
    if (rc != RT_OK) return rc;
    if (job.tile_count > 1) return fail(RT_ERR_INVALID, "rt_render_multi shards the image itself: RT_RENDER_TILE_SHARD must not be set");
    const auto t0 = std::chrono::steady_clock::now();
    DeviceGuard guard(s->dev.device);
    const size_t n = (size_t)job.width * job.height * 3;
    if ((rc = ensure_out_buffers(s, n)) != RT_OK) return rc;
    if ((rc = ensure_replicas(s, n_gpus, n)) != RT_OK) return rc;
    const RenderTuning tune = tuning_for(s, cfg);
    // shard g: the g-th of N equal ranges of the paths (sample-major: sample ranges of every pixel, cut evenly), or every sample of the 4-row bands b with b % N == g
    std::vector<RenderJob> jobs((size_t)n_gpus, job);
    const int32_t S = job.sample_end - job.sample_begin;
    for (int g = 0; g < n_gpus; ++g) {
        if (shard_mode == RT_SHARD_SAMPLES) { // an even share of the paths in sample-major order: whole samples plus a partial first / last one
            const uint64_t T = (uint64_t)job.width * (uint64_t)job.rows * (uint64_t)S;
            jobs[(size_t)g].path_begin = T * (uint64_t)g / (uint64_t)n_gpus;
            jobs[(size_t)g].path_end = T * (uint64_t)(g + 1) / (uint64_t)n_gpus;
            if (jobs[(size_t)g].path_end == jobs[(size_t)g].path_begin) jobs[(size_t)g].sample_end = jobs[(size_t)g].sample_begin; // nothing for this GPU
        } else {
            jobs[(size_t)g].tile_rank = g;
            jobs[(size_t)g].tile_count = n_gpus;
        }
    }
    std::vector<rt_stats> st((size_t)n_gpus);
    std::vector<cudaError_t> errs((size_t)n_gpus, cudaSuccess);
    auto run = [&](int g) {
        rt_stats& out = st[(size_t)g];
        std::memset(&out, 0, sizeof out);
        cudaError_t e;
        if (g == 0) {
            RenderBuffers& o = s->out;
            if ((e = cudaSetDevice(s->dev.device)) == cudaSuccess && (e = cudaMemsetAsync(o.d_accum, 0, n * sizeof(int64_t), o.stream)) == cudaSuccess)
                e = launch_render(s->dev.scene, jobs[0], tune, o.d_accum, o.stream, &out, &s->workspace);
        } else {
            Replica& r = s->replicas[(size_t)g - 1];
            if ((e = cudaSetDevice(r.device)) == cudaSuccess && (e = cudaMemsetAsync(r.d_accum, 0, n * sizeof(int64_t), r.stream)) == cudaSuccess)
                e = launch_render(r.scene, jobs[(size_t)g], tune, r.d_accum, r.stream, &out, &r.workspace);
        }
        errs[(size_t)g] = e;
    };
    {
        std::vector<std::thread> pool;
        for (int g = 1; g < n_gpus; ++g) pool.emplace_back(run, g);
        run(0); // launch_render returns after its stream has drained
        for (std::thread& th : pool) th.join();
    }
    cudaSetDevice(s->dev.device);
    for (int g = 0; g < n_gpus; ++g)
        if (errs[(size_t)g] != cudaSuccess) return fail_cuda(errs[(size_t)g], "render (multi-GPU shard)");
    AccumShards sh;
    std::memset(&sh, 0, sizeof sh);
    sh.n = n_gpus;
    sh.p[0] = s->out.d_accum;
    for (int g = 1; g < n_gpus; ++g) {
        Replica& r = s->replicas[(size_t)g - 1];
        if (r.peer_ok) {
            sh.p[g] = r.d_accum;
        } else {
            const cudaError_t e = cudaMemcpyPeerAsync(r.d_stage, s->dev.device, r.d_accum, r.device, n * sizeof(int64_t), s->out.stream);
            if (e != cudaSuccess) return fail_cuda(e, "peer copy");
            sh.p[g] = r.d_stage;
        }
    }
    if ((rc = gather_and_copy_out(s, sh, job, out_screen, out_accum)) != RT_OK) return rc;
    if (stats) {
        *stats = st[0];
        for (int g = 1; g < n_gpus; ++g) add_stats(*stats, st[(size_t)g], true); // ms_device: the slowest shard
        stats->kernel_launches += 1; // k_reduce_resolve
        stats->ms_total = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    }
    return RT_OK;
}

// ---- adaptive sampling on one GPU or several (rt_render_adaptive, rt_render_adaptive_multi)
namespace {

// Where the render threads of rt_render_adaptive_multi meet once per check point.  The workers (GPUs 1..n-1) arrive when their rounds
// up to the check point have drained and wait until the calling thread (GPU 0) has run the check and handed out the next list.
// fail() lets every thread go for good: the first error anywhere ends the call without leaving a thread waiting.
class RoundBarrier {
  public:
    explicit RoundBarrier(int workers) : workers_(workers) {}
    bool arrive_and_wait() { // worker; false: stop
        std::unique_lock<std::mutex> lk(m_);
        if (failed_) return false;
        const uint64_t gen = gen_;
        ++arrived_;
        cv_.notify_all();
        cv_.wait(lk, [&] { return gen_ != gen || failed_; });
        return !failed_;
    }
    bool gather() { // GPU 0; false: a worker failed
        std::unique_lock<std::mutex> lk(m_);
        cv_.wait(lk, [&] { return arrived_ == workers_ || failed_; });
        return !failed_;
    }
    void release() {
        std::lock_guard<std::mutex> lk(m_);
        arrived_ = 0;
        ++gen_;
        cv_.notify_all();
    }
    void fail() {
        std::lock_guard<std::mutex> lk(m_);
        failed_ = true;
        cv_.notify_all();
    }
    bool failed() {
        std::lock_guard<std::mutex> lk(m_);
        return failed_;
    }

  private:
    std::mutex m_;
    std::condition_variable cv_;
    int workers_, arrived_ = 0;
    uint64_t gen_ = 0;
    bool failed_ = false;
};

// The rounds of rt_render_adaptive spread over n_gpus GPUs (n_gpus = 1: the scene's own GPU only, with the launches of a plain
// single-GPU render).  GPU g renders the g-th of n_gpus even ranges of each round's paths (sample-major over the active list) into its
// own A or B, on its own host thread; GPU 0 runs the check points and the resolve over every GPU's A and B.
int32_t render_adaptive(rt_scene* s, const rt_render_config* cfg, const rt_adaptive_config* ac, int32_t n_gpus, double* out_screen,
                        int64_t* out_accum, int32_t* out_samples, rt_stats* stats) {
    CHECK_SCENE(s);
    if (!cfg) return fail(RT_ERR_INVALID, "null config");
    // argument checks first: they need no committed scene
    if (!ac) return fail(RT_ERR_INVALID, "null adaptive config");
    if (ac->step < 1) return fail(RT_ERR_INVALID, "adaptive step < 1");
    if (!(ac->threshold >= 0.0) || !std::isfinite(ac->threshold)) return fail(RT_ERR_INVALID, "adaptive threshold must be finite and >= 0");
    if (ac->radius < 0 || ac->radius > 8) return fail(RT_ERR_INVALID, "adaptive radius outside 0..8");
    if (ac->min_samples < 0 || ac->min_samples > cfg->samples_per_pixel) return fail(RT_ERR_INVALID, "adaptive min_samples outside 0..samples_per_pixel");
    if (RT_RENDER_TILE_COUNT(cfg->flags) > 1 || (cfg->flags & RT_RENDER_NO_WAIT))
        return fail(RT_ERR_INVALID, "rt_render_adaptive takes neither a tile shard (RT_RENDER_TILE_SHARD with count > 1) nor RT_RENDER_NO_WAIT");
    if (cfg->sample_begin != 0 || (cfg->sample_end != 0 && cfg->sample_end != cfg->samples_per_pixel))
        return fail(RT_ERR_INVALID, "rt_render_adaptive renders every sample range itself: sample_begin / sample_end must cover [0, samples_per_pixel)");
    if (n_gpus < 1 || n_gpus > RT_MAX_GPUS) return fail(RT_ERR_INVALID, "n_gpus outside 1..16");
    RenderJob job;
    int32_t rc = make_job(s, cfg, job);
    if (rc != RT_OK) return rc;
    const auto t0 = std::chrono::steady_clock::now();
    DeviceGuard guard(s->dev.device);
    const size_t npix = (size_t)job.width * job.height, n = npix * 3;
    // A replica's B starts nb elements after its A: an even offset keeps B 16-byte aligned for the kernels' 128-bit loads when n is odd
    const size_t nb = (n + 1) & ~(size_t)1;
    if ((rc = ensure_out_buffers(s, n)) != RT_OK) return rc;
    if ((rc = ensure_adaptive_buffers(s, npix)) != RT_OK) return rc;
    if (n_gpus > 1) {
        if ((rc = ensure_replicas(s, n_gpus, 2 * nb)) != RT_OK) return rc; // d_accum = A | B, d_stage (no P2P route) as large
        for (int g = 1; g < n_gpus; ++g) {
            Replica& r = s->replicas[(size_t)g - 1];
            if (npix <= r.list_cap) continue;
            cudaError_t e;
            if ((e = cudaSetDevice(r.device)) == cudaSuccess) {
                if (r.d_list) cudaFree(r.d_list);
                r.d_list = nullptr; r.list_cap = 0;
                e = cudaMalloc(&r.d_list, npix * sizeof(uint32_t));
            }
            cudaSetDevice(s->dev.device);
            if (e != cudaSuccess) return fail_cuda(e, "replica pixel list");
            r.list_cap = npix;
        }
    }
    RenderBuffers& o = s->out;
    AdaptiveBuffers& b = s->adaptive;
    const RenderTuning tune = tuning_for(s, cfg);
    const int32_t max = job.spp_total, step = ac->step;
    const uint32_t rendered = (uint32_t)job.width * (uint32_t)job.rows;
    cudaError_t e;
    if ((e = cudaMemsetAsync(b.d_a, 0, n * sizeof(int64_t), o.stream)) != cudaSuccess || (e = cudaMemsetAsync(b.d_b, 0, n * sizeof(int64_t), o.stream)) != cudaSuccess ||
        (e = cudaMemsetAsync(b.d_samples, 0, npix * sizeof(int32_t), o.stream)) != cudaSuccess || (e = launch_adaptive_iota(b.d_list[0], rendered, o.stream)) != cudaSuccess)
        return fail_cuda(e, "adaptive set-up");

    // every GPU's A and B as GPU 0 reads them: in place (its own, P2P-mapped peers, alias mode) or copied into staging next to it
    auto shards = [&](AdaptiveShards& sh) -> cudaError_t {
        std::memset(&sh, 0, sizeof sh);
        sh.n = n_gpus;
        sh.a[0] = b.d_a; sh.b[0] = b.d_b;
        for (int g = 1; g < n_gpus; ++g) {
            Replica& r = s->replicas[(size_t)g - 1];
            const int64_t* ab = r.d_accum;
            if (!r.peer_ok) {
                const cudaError_t ce = cudaMemcpyPeerAsync(r.d_stage, s->dev.device, r.d_accum, r.device, 2 * nb * sizeof(int64_t), o.stream);
                if (ce != cudaSuccess) return ce;
                ab = r.d_stage;
            }
            sh.a[g] = ab; sh.b[g] = ab + nb;
        }
        return cudaSuccess;
    };

    std::vector<std::vector<rt_stats>> st((size_t)n_gpus); // [GPU][round]
    std::vector<cudaError_t> errs((size_t)n_gpus, cudaSuccess);
    std::vector<const char*> what((size_t)n_gpus, "");
    RoundBarrier bar(n_gpus - 1);
    uint32_t n_active = rendered; // written by GPU 0 at a check point, read by the workers once the barrier lets them go
    int cur = 0;                  // GPU 0's current list (b.d_list[cur]); the workers' is r.d_list
    auto run = [&](int g) {
        Replica* r = g ? &s->replicas[(size_t)g - 1] : nullptr;
        cudaStream_t stream = r ? r->stream : o.stream;
        int64_t* A = r ? r->d_accum : b.d_a;
        int64_t* B = r ? r->d_accum + nb : b.d_b;
        cudaError_t& err = errs[(size_t)g];
        auto stop = [&](cudaError_t ce, const char* w) { err = ce; what[(size_t)g] = w; bar.fail(); };
        if (r && ((err = cudaSetDevice(r->device)) != cudaSuccess || (err = cudaMemsetAsync(r->d_accum, 0, 2 * nb * sizeof(int64_t), stream)) != cudaSuccess ||
                  (err = launch_adaptive_iota(r->d_list, rendered, stream)) != cudaSuccess))
            return stop(err, "adaptive set-up");
        uint32_t na = rendered;
        for (int64_t k = 0; na > 0 && k * step < max; ++k) {
            if (n_gpus > 1 && bar.failed()) return;
            const int32_t s0 = (int32_t)(k * step), s1 = (int32_t)std::min<int64_t>((k + 1) * step, max);
            RenderJob rj = job;
            rj.sample_begin = s0; rj.sample_end = s1;
            rj.d_pixels = r ? r->d_list : b.d_list[cur]; rj.n_pixels = na;
            // an even share of the round's paths: balanced in every round, consecutive paths on neighbouring pixels
            const uint64_t T = (uint64_t)na * (uint64_t)(s1 - s0);
            rj.path_begin = T * (uint64_t)g / (uint64_t)n_gpus;
            rj.path_end = T * (uint64_t)(g + 1) / (uint64_t)n_gpus;
            rt_stats rs;
            std::memset(&rs, 0, sizeof rs);
            if (rj.path_end > rj.path_begin) { // an empty range renders nothing (more GPUs than paths)
                const DeviceScene& scene = r ? r->scene : s->dev.scene;
                if ((err = launch_render(scene, rj, tune, (k & 1) ? B : A, stream, &rs, r ? &r->workspace : &s->workspace)) != cudaSuccess)
                    return stop(err, "adaptive render round");
            }
            st[(size_t)g].push_back(rs);
            if (!(k & 1) || s1 < ac->min_samples || s1 >= max) continue;
            if (r) { // launch_render has drained the stream, except where the range was empty: the set-up may still be in flight
                if ((err = cudaStreamSynchronize(stream)) != cudaSuccess) return stop(err, "adaptive round sync");
                if (!bar.arrive_and_wait()) return;
                na = n_active;
                continue;
            }
            if (!bar.gather()) return;
            AdaptiveCheck c;
            if ((err = shards(c.shards)) != cudaSuccess) return stop(err, "peer copy");
            c.d_list_in = b.d_list[cur]; c.n_active = na; c.d_list_out = b.d_list[cur ^ 1]; c.count_out = b.h_count;
            c.d_u = b.d_u; c.d_keep = b.d_keep; c.d_samples = b.d_samples;
            c.d_temp = b.d_temp; c.temp_bytes = b.temp_bytes;
            c.W = job.width; c.rows = job.rows; c.n = s1; c.radius = ac->radius; c.threshold = ac->threshold;
            if ((err = launch_adaptive_check(c, o.stream)) != cudaSuccess) return stop(err, "adaptive check");
            if ((err = cudaStreamSynchronize(o.stream)) != cudaSuccess) return stop(err, "adaptive check sync");
            na = n_active = *b.h_count;
            cur ^= 1;
            if (n_gpus > 1) {
                for (int h = 1; h < n_gpus && na > 0; ++h) {
                    Replica& rh = s->replicas[(size_t)h - 1];
                    if ((err = cudaMemcpyPeerAsync(rh.d_list, rh.device, b.d_list[cur], s->dev.device, na * sizeof(uint32_t), o.stream)) != cudaSuccess)
                        return stop(err, "pixel list copy");
                }
                if ((err = cudaStreamSynchronize(o.stream)) != cudaSuccess) return stop(err, "pixel list copy sync");
                bar.release();
            }
        }
        if (r && (err = cudaStreamSynchronize(stream)) != cudaSuccess) return stop(err, "adaptive round sync");
    };
    {
        std::vector<std::thread> pool;
        bool started = true;
        try {
            for (int g = 1; g < n_gpus; ++g) pool.emplace_back(run, g);
        } catch (const std::system_error&) {
            started = false;
            bar.fail();
        }
        if (started) run(0); // the calling thread is GPU 0
        for (std::thread& th : pool) th.join();
        if (!started) return fail(RT_ERR_CUDA, "could not start the render threads");
    }
    for (int g = 0; g < n_gpus; ++g)
        if (errs[(size_t)g] != cudaSuccess) return fail_cuda(errs[(size_t)g], what[(size_t)g]);
    AdaptiveShards sh;
    if ((e = launch_adaptive_fill(b.d_list[cur], n_active, max, b.d_samples, o.stream)) != cudaSuccess) return fail_cuda(e, "adaptive counts");
    if ((e = shards(sh)) != cudaSuccess) return fail_cuda(e, "peer copy");
    if ((e = launch_resolve_adaptive(sh, b.d_samples, o.d_accum, o.d_u8, job.width, job.height, o.stream)) != cudaSuccess) return fail_cuda(e, "adaptive resolve");
    if (out_screen && (e = cudaMemcpyAsync(o.h_u8, o.d_u8, n, cudaMemcpyDeviceToHost, o.stream)) != cudaSuccess) return fail_cuda(e, "screen copy");
    if (out_accum && (e = cudaMemcpyAsync(out_accum, o.d_accum, n * sizeof(int64_t), cudaMemcpyDeviceToHost, o.stream)) != cudaSuccess) return fail_cuda(e, "accum copy");
    if (out_samples && (e = cudaMemcpyAsync(out_samples, b.d_samples, npix * sizeof(int32_t), cudaMemcpyDeviceToHost, o.stream)) != cudaSuccess)
        return fail_cuda(e, "samples copy");
    if ((e = cudaStreamSynchronize(o.stream)) != cudaSuccess) return fail_cuda(e, "adaptive sync");
    if (out_screen) widen_screen(o.h_u8, out_screen, n);
    if (stats) { // the GPUs of a round run at the same time, the rounds one after the other
        std::memset(stats, 0, sizeof *stats);
        for (size_t k = 0; k < st[0].size(); ++k) {
            rt_stats round = st[0][k];
            for (int g = 1; g < n_gpus; ++g) add_stats(round, st[(size_t)g][k], true);
            add_stats(*stats, round, false);
        }
        stats->ms_total = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    }
    return RT_OK;
}

} // namespace

int32_t rt_render_adaptive(rt_scene* s, const rt_render_config* cfg, const rt_adaptive_config* ac, double* out_screen, int64_t* out_accum,
                           int32_t* out_samples, rt_stats* stats) {
    return render_adaptive(s, cfg, ac, 1, out_screen, out_accum, out_samples, stats);
}

int32_t rt_render_adaptive_multi(rt_scene* s, const rt_render_config* cfg, const rt_adaptive_config* ac, int32_t n_gpus, double* out_screen,
                                 int64_t* out_accum, int32_t* out_samples, rt_stats* stats) {
    return render_adaptive(s, cfg, ac, n_gpus, out_screen, out_accum, out_samples, stats);
}

// ---- peer group: the exchange of the one-process-per-GPU layout without a collective library on the data path
struct rt_peer_group {
    int32_t rank = 0, world = 1;
    int64_t n_elems = 0;
    char* base = nullptr;                 // own allocation: n_elems int64 + one 256-byte flag block
    std::vector<char*> peer;              // every rank's allocation as mapped here (own slot = base)
    uint32_t step = 0;                    // steps published by this rank so far
    uint32_t* d_timeout = nullptr;
    bool connected = false;
    int64_t* accum(int r) const { return reinterpret_cast<int64_t*>(peer[(size_t)r]); }
    uint32_t* published(int r) const { return reinterpret_cast<uint32_t*>(peer[(size_t)r] + (size_t)n_elems * sizeof(int64_t)); }
    uint32_t* consumed(int r) const { return published(r) + 16; } // its own 64-byte line
};

rt_peer_group* rt_peer_create(int32_t rank, int32_t world, int64_t n_elems, uint8_t out_handle[RT_PEER_HANDLE_BYTES]) {
    if (rank < 0 || world < 1 || rank >= world || world > RT_MAX_GPUS || n_elems <= 0 || !out_handle) { fail(RT_ERR_INVALID, "bad peer group request"); return nullptr; }
    static_assert(sizeof(cudaIpcMemHandle_t) <= RT_PEER_HANDLE_BYTES, "handle size");
    rt_peer_group* g = new rt_peer_group();
    g->rank = rank; g->world = world; g->n_elems = n_elems;
    const size_t bytes = (size_t)n_elems * sizeof(int64_t) + 256;
    cudaError_t e = cudaMalloc(&g->base, bytes);
    if (e == cudaSuccess) e = cudaMemset(g->base, 0, bytes);
    if (e == cudaSuccess) e = cudaMalloc(&g->d_timeout, sizeof(uint32_t));
    if (e == cudaSuccess) e = cudaMemset(g->d_timeout, 0, sizeof(uint32_t));
    cudaIpcMemHandle_t h;
    if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, g->base);
    if (e != cudaSuccess) { fail_cuda(e, "peer group allocation"); rt_peer_destroy(g); return nullptr; }
    std::memset(out_handle, 0, RT_PEER_HANDLE_BYTES);
    std::memcpy(out_handle, &h, sizeof h);
    g->peer.assign((size_t)world, nullptr);
    g->peer[(size_t)rank] = g->base;
    return g;
}

int32_t rt_peer_connect(rt_peer_group* g, const uint8_t* all_handles) {
    if (!g || !all_handles) return fail(RT_ERR_INVALID, "null peer group");
    for (int r = 0; r < g->world; ++r) {
        if (r == g->rank || g->peer[(size_t)r]) continue;
        cudaIpcMemHandle_t h;
        std::memcpy(&h, all_handles + (size_t)r * RT_PEER_HANDLE_BYTES, sizeof h);
        void* p = nullptr;
        const cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) return fail_cuda(e, "cudaIpcOpenMemHandle (peer accumulator)");
        g->peer[(size_t)r] = static_cast<char*>(p);
    }
    g->connected = true;
    return RT_OK;
}

int64_t* rt_peer_accum(rt_peer_group* g) { return g ? reinterpret_cast<int64_t*>(g->base) : nullptr; }

int32_t rt_peer_begin(rt_peer_group* g, void* cuda_stream) {
    if (!g || !g->connected) return fail(RT_ERR_STATE, "peer group not connected");
    cudaStream_t st = (cudaStream_t)cuda_stream;
    cudaError_t e = cudaSuccess;
    // the gatherer (rank 0) must have read the previous step's sums before they are cleared
    if (g->rank != 0 && g->step > 0) e = launch_flag_wait(g->consumed(0), g->step, g->d_timeout, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(g->base, 0, (size_t)g->n_elems * sizeof(int64_t), st);
    if (e != cudaSuccess) return fail_cuda(e, "peer begin");
    return RT_OK;
}

int32_t rt_peer_publish(rt_peer_group* g, void* cuda_stream) {
    if (!g || !g->connected) return fail(RT_ERR_STATE, "peer group not connected");
    ++g->step;
    const cudaError_t e = launch_flag_publish(g->published(g->rank), g->step, (cudaStream_t)cuda_stream);
    if (e != cudaSuccess) return fail_cuda(e, "peer publish");
    return RT_OK;
}

int32_t rt_peer_gather_resolve(rt_peer_group* g, double* d_screen, int32_t width, int32_t height, int32_t spp, int32_t rendered_rows, void* cuda_stream) {
    if (!g || !g->connected) return fail(RT_ERR_STATE, "peer group not connected");
    if (g->rank != 0) return fail(RT_ERR_STATE, "rank 0 gathers");
    if (!d_screen || width <= 0 || height <= 0 || spp <= 0 || (int64_t)width * height * 3 != g->n_elems) return fail(RT_ERR_INVALID, "bad gather arguments");
    if (g->step == 0) return fail(RT_ERR_STATE, "rt_peer_publish first");
    AccumShards sh;
    std::memset(&sh, 0, sizeof sh);
    sh.n = g->world;
    sh.need = g->step;
    sh.timeout_flag = g->d_timeout;
    for (int r = 0; r < g->world; ++r) { sh.p[r] = g->accum(r); sh.ready[r] = g->published(r); }
    cudaStream_t st = (cudaStream_t)cuda_stream;
    cudaError_t e = launch_reduce_resolve(sh, nullptr, nullptr, d_screen, width, height, spp, rendered_rows, st);
    if (e == cudaSuccess) e = launch_flag_publish(g->consumed(0), g->step, st); // the peers may clear their accumulators now
    if (e != cudaSuccess) return fail_cuda(e, "peer gather");
    return RT_OK;
}

int32_t rt_peer_timed_out(rt_peer_group* g) {
    if (!g) return RT_ERR_INVALID;
    uint32_t v = 0;
    if (cudaMemcpy(&v, g->d_timeout, sizeof v, cudaMemcpyDeviceToHost) != cudaSuccess) return RT_ERR_CUDA;
    return (int32_t)v;
}

void rt_peer_destroy(rt_peer_group* g) {
    if (!g) return;
    for (int r = 0; r < (int)g->peer.size(); ++r)
        if (r != g->rank && g->peer[(size_t)r]) cudaIpcCloseMemHandle(g->peer[(size_t)r]);
    if (g->base) cudaFree(g->base);
    if (g->d_timeout) cudaFree(g->d_timeout);
    delete g;
}

int32_t rt_write_ppm(const char* path, const double* screen, int32_t width, int32_t height) {
    if (!screen || width <= 0 || height <= 0) return fail(RT_ERR_INVALID, "bad screen");
    std::string err;
    if (!write_ppm_p3(path, screen, width, height, err)) return fail(RT_ERR_IO, err);
    return RT_OK;
}

int32_t rt_write_ppm_binary(const char* path, const double* screen, int32_t width, int32_t height) {
    if (!screen || width <= 0 || height <= 0) return fail(RT_ERR_INVALID, "bad screen");
    std::string err;
    if (!write_ppm_p6(path, screen, width, height, err)) return fail(RT_ERR_IO, err);
    return RT_OK;
}
int32_t rt_write_ply_binary(const char* path, const double* verts, int64_t nv, const uint32_t* idx, int64_t nt) {
    if (!path || !verts || !idx || nv <= 0 || nt <= 0) return fail(RT_ERR_INVALID, "bad mesh");
    std::vector<double> v(verts, verts + 3 * nv);
    std::vector<uint32_t> f(idx, idx + 3 * nt);
    std::string err;
    if (!write_ply_binary(path, v, f, err)) return fail(RT_ERR_IO, err);
    return RT_OK;
}
int32_t rt_ply_convert_binary(const char* ascii_path, const char* binary_path) {
    if (!ascii_path || !binary_path) return fail(RT_ERR_INVALID, "null path");
    std::vector<double> v; std::vector<uint32_t> f;
    std::string err;
    if (!read_ply_any(ascii_path, 1.0, v, f, err) || !write_ply_binary(binary_path, v, f, err)) return fail(RT_ERR_IO, err);
    return RT_OK;
}

#define PFX(name) rt_##name
// render_scene_with_time (world.rs:1249-1330)
int32_t PFX(render_scene_with_time)(rt_scene* s, double t0, double t1, const char* path, const rt_render_config* cfg_in, double* out_screen, rt_stats* stats) {
    CHECK_SCENE(s);
    rt_render_config cfg;
    if (cfg_in) {
        cfg = *cfg_in;
    } else {
        std::memset(&cfg, 0, sizeof cfg);
        cfg.image_width = 500; cfg.aspect_ratio = 1.0; cfg.samples_per_pixel = 500; cfg.max_depth = 50; // world.rs:1253-1257
        cfg.compat_threads = 11;                                                                          // world.rs:18, 1281
        cfg.seed = 1;
    }
    const double lookfrom[3] = {13, 2, 3}, lookat[3] = {0, 0, 0}, vup[3] = {0, 1, 0}, bg[3] = {0.7, 0.8, 1.0}; // world.rs:1252, 1259-1263
    int32_t rc = PFX(scene_set_camera)(s, lookfrom, lookat, vup, 20.0, cfg.aspect_ratio, 0.1, 10.0, t0, t1);
    if (rc != RT_OK) return rc;
    if ((rc = PFX(scene_set_background)(s, bg)) != RT_OK) return rc;
    if ((rc = PFX(scene_commit)(s)) != RT_OK) return rc;
    const int32_t H = PFX(image_height)(&cfg);
    if (H <= 0) return fail(RT_ERR_INVALID, "image height <= 0");
    std::vector<double> local;
    double* screen = out_screen;
    if (!screen) { local.resize((size_t)cfg.image_width * H * 3); screen = local.data(); }
    if ((rc = PFX(render)(s, &cfg, screen, nullptr, stats)) != RT_OK) return rc;
    if (path) return PFX(write_ppm)(path, screen, cfg.image_width, H);
    return RT_OK;
}
#undef PFX

// ---------------------------------------------------------------- parity hook
int32_t rt_trace_batch(rt_scene* s, const rt_ray* rays, int64_t n, double t_min, double t_max, int32_t flags, uint64_t seed, rt_hit* out) {
    CHECK_SCENE(s);
    if (!s->committed || !s->dev.valid) return fail(RT_ERR_STATE, "scene not committed");
    if (n < 0 || (n > 0 && (!rays || !out))) return fail(RT_ERR_INVALID, "bad batch");
    if (n == 0) return RT_OK;
    // the f32 slab test is conservative for origins inside the committed domain and for times inside
    // the span the moving bounds were built for
    const double lim = 4.0 * s->domain_radius;
    bool has_moving = false;
    for (const Node& nd : s->nodes) has_moving = has_moving || nd.kind == N_MOVING || nd.kind == N_GRAVITY;
    for (int64_t i = 0; i < n; ++i) {
        for (int a = 0; a < 3; ++a)
            if (!(std::fabs(rays[i].o[a]) <= lim)) return fail(RT_ERR_INVALID, "ray origin outside the committed scene domain (4x the scene radius)");
        if (has_moving && !(rays[i].time >= s->span0 - 1e-12 && rays[i].time <= s->span1 + 1e-12))
            return fail(RT_ERR_INVALID, "ray time outside the camera shutter the moving-primitive bounds were built for");
    }
    rt_ray* d_rays = nullptr;
    rt_hit* d_out = nullptr;
    cudaError_t e;
    int32_t rc = RT_OK;
    do {
        if ((e = cudaMalloc(&d_rays, (size_t)n * sizeof(rt_ray))) != cudaSuccess) { rc = fail_cuda(e, "ray allocation"); break; }
        if ((e = cudaMalloc(&d_out, (size_t)n * sizeof(rt_hit))) != cudaSuccess) { rc = fail_cuda(e, "hit allocation"); break; }
        if ((e = cudaMemcpy(d_rays, rays, (size_t)n * sizeof(rt_ray), cudaMemcpyHostToDevice)) != cudaSuccess) { rc = fail_cuda(e, "ray upload"); break; }
        if ((e = launch_trace_batch(s->dev.scene, d_rays, n, t_min, t_max, flags, seed, d_out, nullptr)) != cudaSuccess) { rc = fail_cuda(e, "trace launch"); break; }
        if ((e = cudaMemcpy(out, d_out, (size_t)n * sizeof(rt_hit), cudaMemcpyDeviceToHost)) != cudaSuccess) { rc = fail_cuda(e, "hit download"); break; }
    } while (0);
    if (d_rays) cudaFree(d_rays);
    if (d_out) cudaFree(d_out);
    return rc;
}

// unit-level device checks (tests only; see kernels.h launch_unit_op)
RTB_EXPORT int32_t rt_unit_op(rt_scene* s, int32_t op, uint32_t ia, uint32_t ib, uint32_t ic, uint32_t id, const double* in8, double* out8) {
    CHECK_SCENE(s);
    if (!s->committed || !s->dev.valid) return fail(RT_ERR_STATE, "scene not committed");
    const cudaError_t e = launch_unit_op(s->dev.scene, op, ia, ib, ic, id, in8, out8);
    if (e != cudaSuccess) return fail_cuda(e, "unit op");
    return RT_OK;
}

// Host-only validation of the flattener + BVH builder (no CUDA): checks that every leaf primitive's
// bounds lie inside its leaf box and every node inside its parent, that each typed slot is referenced
// by exactly one leaf, and returns out[0] nodes, [1] max depth, [2] main instances, [3] all instances,
// [4] media, [5..10] primitives per type, [11] leaves, [12] violations (0 = valid), [13] prims numbered.
RTB_EXPORT int32_t rt_debug_host_scene(rt_scene* s, void* out_scene, uint64_t out_bytes) {
    CHECK_SCENE(s);
    if (!out_scene || out_bytes != sizeof(DeviceScene)) return fail(RT_ERR_INVALID, "out_scene must hold one DeviceScene (csrc/rt_types.h)");
    std::shared_ptr<HostFlat> hf = std::make_shared<HostFlat>();
    const int32_t fr = flatten_host(s, *hf);
    if (fr != RT_OK) return fr;
    HostFlat& HF = *hf;
    DeviceScene D;
    std::memset(&D, 0, sizeof D);
    D.nodes = HF.nodes.data(); D.mnodes = HF.mnodes.empty() ? nullptr : HF.mnodes.data(); D.nodes4 = HF.nodes4.empty() ? nullptr : HF.nodes4.data(); D.mnodes4 = HF.mnodes4.empty() ? nullptr : HF.mnodes4.data();
    D.spheres = HF.spheres.data(); D.movings = HF.movings.data(); D.gravities = HF.gravities.data(); D.gravity_table = HF.gtable.data();
    D.rects = HF.rects.data(); D.boxes = HF.boxes.data(); D.tris = HF.tris.data();
    for (int t = 0; t < (int)PRIM_TYPE_COUNT; ++t) D.meta[t] = HF.meta[t].data();
    D.instances = HF.instances.data(); D.ops = HF.ops.data(); D.media = HF.media.data(); D.materials = HF.dmats.data(); D.textures = HF.dtex.data();
    D.perlin = HF.perlin.data(); D.texels = HF.texels.data();
    set_scene_scalars(s, HF, D);
    std::memcpy(out_scene, &D, sizeof D);
    s->debug_flat = hf; // the arrays live until the next call or rt_scene_destroy
    return RT_OK;
}

RTB_EXPORT int32_t rt_scene_host_check(rt_scene* s, int64_t out[16]) {
    CHECK_SCENE(s);
    if (!out) return fail(RT_ERR_INVALID, "null out");
    HostFlat HF;
    const int32_t fr = flatten_host(s, HF);
    if (fr != RT_OK) return fr;
    for (int i = 0; i < 16; ++i) out[i] = 0;
    out[0] = (int64_t)HF.nodes.size(); out[1] = HF.max_depth; out[2] = HF.n_main_instances; out[3] = (int64_t)HF.instances.size();
    out[4] = (int64_t)HF.media.size();
    const size_t counts[PRIM_TYPE_COUNT] = {HF.spheres.size(), HF.movings.size(), HF.gravities.size(), HF.rects.size(), HF.boxes.size(), HF.tris.size()};
    for (int t = 0; t < (int)PRIM_TYPE_COUNT; ++t) out[5 + t] = (int64_t)counts[t];
    std::vector<std::vector<uint8_t>> seen(PRIM_TYPE_COUNT);
    for (int t = 0; t < (int)PRIM_TYPE_COUNT; ++t) seen[(size_t)t].assign(counts[t], 0);
    int64_t violations = 0, leaves = 0;
    for (const Instance& in : HF.instances) {
        struct Item { uint32_t node; float mn[3], mx[3]; };
        std::vector<Item> st;
        Item r; r.node = in.root;
        for (int a = 0; a < 3; ++a) { r.mn[a] = -INFINITY; r.mx[a] = INFINITY; }
        st.push_back(r);
        while (!st.empty()) {
            const Item it = st.back();
            st.pop_back();
            const BvhNode32& nd = HF.nodes[it.node];
            for (int a = 0; a < 3; ++a)
                if (nd.min[a] < it.mn[a] || nd.max[a] > it.mx[a] || !(nd.min[a] <= nd.max[a])) ++violations;
            if (nd.count) {
                ++leaves;
                const uint32_t type = (nd.count >> 24) & 0x7fu, n = nd.count & 0xffffffu;
                for (uint32_t i = nd.first; i < nd.first + n; ++i) {
                    if (type >= PRIM_TYPE_COUNT || i >= counts[type]) { ++violations; continue; }
                    if (seen[type][i]++) ++violations;
                    double mn[3], mx[3];
                    bool have = true;
                    switch (type) {
                    case PRIM_SPHERE: { const DSphere& q = HF.spheres[i]; const double c[3] = {q.cx, q.cy, q.cz}; for (int a = 0; a < 3; ++a) { mn[a] = c[a] - std::fabs(q.r); mx[a] = c[a] + std::fabs(q.r); } } break;
                    case PRIM_RECT: { const DRect& q = HF.rects[i]; const int ax = q.axis, ia = ax == 0 ? 1 : 0, ib = ax == 2 ? 1 : 2; mn[ax] = mx[ax] = q.k; mn[ia] = q.a0; mx[ia] = q.a1; mn[ib] = q.b0; mx[ib] = q.b1; } break;
                    case PRIM_BOX: { const DBox& q = HF.boxes[i]; for (int a = 0; a < 3; ++a) { mn[a] = std::fmin(q.p0[a], q.p1[a]); mx[a] = std::fmax(q.p0[a], q.p1[a]); } } break;
                    case PRIM_TRI: { const DTri& q = HF.tris[i]; for (int a = 0; a < 3; ++a) { mn[a] = std::fmin(q.v0[a], std::fmin(q.v1[a], q.v2[a])); mx[a] = std::fmax(q.v0[a], std::fmax(q.v1[a], q.v2[a])); } } break;
                    default: have = false; break;
                    }
                    if (have)
                        for (int a = 0; a < 3; ++a)
                            if (mn[a] < (double)nd.min[a] || mx[a] > (double)nd.max[a]) ++violations;
                }
            } else {
                for (uint32_t c = 0; c < 2; ++c) {
                    Item ch; ch.node = nd.first + c;
                    if (ch.node >= HF.nodes.size() || (nd.first & 1u)) { ++violations; continue; }
                    for (int a = 0; a < 3; ++a) { ch.mn[a] = nd.min[a]; ch.mx[a] = nd.max[a]; }
                    st.push_back(ch);
                }
            }
        }
    }
    for (int t = 0; t < (int)PRIM_TYPE_COUNT; ++t)
        for (uint8_t v : seen[(size_t)t])
            if (v != 1) ++violations;
    out[11] = leaves; out[12] = violations; out[13] = s->n_prims;
    out[14] = (int64_t)s->dev.bytes; // bytes uploaded host->device by the last rt_scene_commit
    out[15] = s->dev.device_built_prims; // primitives whose BVH the last rt_scene_commit built on the device
    return RT_OK;
}

// wavefront tuning knobs (bench / profiling): wave_slots = resident path slots
RTB_EXPORT int32_t rt_scene_set_bvh_builder(rt_scene* s, int32_t builder) {
    CHECK_SCENE(s);
    if (builder != RT_BVH_HOST_SAH && builder != RT_BVH_DEVICE_LBVH) return fail(RT_ERR_INVALID, "unknown BVH builder");
    s->tuning.bvh_builder = builder;
    return RT_OK;
}

RTB_EXPORT int32_t rt_scene_set_bvh_width(rt_scene* s, int32_t width) {
    CHECK_SCENE(s);
    if (width != 0 && width != 2 && width != 4) return fail(RT_ERR_INVALID, "BVH width must be 0 (auto), 2 or 4");
    s->tuning.bvh_wide = width == 4 ? 1 : (width == 2 ? 0 : -1);
    s->committed = false;
    return RT_OK;
}

RTB_EXPORT int32_t rt_scene_bvh_width(rt_scene* s) {
    CHECK_SCENE(s);
    if (!s->committed || !s->dev.valid) return fail(RT_ERR_STATE, "scene not committed");
    return s->dev.scene.nodes4 ? 4 : 2;
}

RTB_EXPORT int32_t rt_scene_set_tuning(rt_scene* s, uint32_t wave_slots) {
    CHECK_SCENE(s);
    if (wave_slots) s->tuning.wave_slots = wave_slots < 128 ? 128 : wave_slots;
    return RT_OK;
}

} // extern "C"
