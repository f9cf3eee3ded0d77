// rt_device.cuh — device-side restatement of the reference hot path for sm_100a.
//
//   vec3.rs / ray.rs           -> D3 / Ray (f64)
//   aabb.rs + bvh.rs           -> slab2() + trace_instance(): f32 slab test of sibling pairs fetched
//                                 with two 128-bit read-only loads per node, short stack, ordered descent
//   hit.rs  Hittable impls     -> hit_sphere / hit_rect / hit_box / hit_tri (f64), finalize_hit()
//   hit.rs  Translate/RotateY  -> xform_ray() going in, chain post-processing coming out (quirks kept)
//   hit.rs  ConstantMedium     -> medium_query()
//   hit.rs  Material impls     -> scatter_*()
//   texture.rs / perlin.rs     -> tex_value() / perlin_noise() / perlin_turbulence()
//   camera.rs                  -> camera_get_ray()
//   rand thread_rng()          -> PathRng (Philox-4x32-10, one counter step per draw)
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../rt_types.h"

namespace rtb {

#define RT_DEV __device__ __forceinline__
#define RT_STACK 64

// ------------------------------------------------------------------ D3 (vec3.rs)
struct D3 {
    double x, y, z;
};
RT_DEV D3 mk3(double x, double y, double z) { D3 r; r.x = x; r.y = y; r.z = z; return r; }
RT_DEV D3 operator+(D3 a, D3 b) { return mk3(a.x + b.x, a.y + b.y, a.z + b.z); }
RT_DEV D3 operator-(D3 a, D3 b) { return mk3(a.x - b.x, a.y - b.y, a.z - b.z); }
RT_DEV D3 operator-(D3 a) { return mk3(-a.x, -a.y, -a.z); }
RT_DEV D3 operator*(D3 a, double s) { return mk3(a.x * s, a.y * s, a.z * s); }
RT_DEV D3 operator*(double s, D3 a) { return mk3(a.x * s, a.y * s, a.z * s); }
RT_DEV double dot(D3 a, D3 b) { return fma(a.z, b.z, fma(a.y, b.y, a.x * b.x)); }
RT_DEV D3 cross(D3 a, D3 b) { return mk3(fma(a.y, b.z, -(a.z * b.y)), fma(a.z, b.x, -(a.x * b.z)), fma(a.x, b.y, -(a.y * b.x))); }
RT_DEV double length_squared(D3 a) { return dot(a, a); }
RT_DEV D3 unit(D3 a) { return a * (1.0 / sqrt(length_squared(a))); }                 // vec3.rs:55-57
RT_DEV D3 reflect(D3 v, D3 n) { const double k = -2.0 * dot(v, n); return mk3(fma(k, n.x, v.x), fma(k, n.y, v.y), fma(k, n.z, v.z)); }                    // vec3.rs:64-66
RT_DEV bool near_zero(D3 a) { const double s = 1e-8; return fabs(a.x) < s && fabs(a.y) < s && fabs(a.z) < s; } // vec3.rs:59-62
RT_DEV D3 refract(D3 uv, D3 n, double etai_over_etat) {                              // vec3.rs:116-121
    const double cos_theta = fmin(dot(-uv, n), 1.0);
    const D3 r_out_perp = etai_over_etat * (uv + cos_theta * n);
    const D3 r_out_parallel = -(sqrt(fabs(1.0 - length_squared(r_out_perp)))) * n;
    return r_out_perp + r_out_parallel;
}
RT_DEV double axis_of(D3 a, int ax) { return ax == 0 ? a.x : (ax == 1 ? a.y : a.z); }

struct Ray { // ray.rs:3-8
    D3 o, d;
    double time;
};
RT_DEV D3 ray_at(const Ray& r, double t) { return mk3(fma(r.d.x, t, r.o.x), fma(r.d.y, t, r.o.y), fma(r.d.z, t, r.o.z)); } // ray.rs:31-33

// Measured on B200 (tools/ab_libs.sh, book-1 final, 500 spp, same box): Philox inlined at its 19 call sites 100.4 ms, one
// out-of-line copy 94.4 ms (the kernel stalled on instruction fetch for 19 % of its samples).  Resolving the samplers'
// draw positions at compile time removes next_u32's word selection but was 1-8 % slower in every combination (fewer
// instructions, slower kernel: at ~11 active lanes per instruction the bound is fetch / issue latency of divergent
// code: four unrolled copies of the candidate).  What did pay, late in round 2, is ONE copy of the candidate that takes its
// two / three words at once and picks them with selects (next2_pm1 / next3_pm1 below): book-1 final 80.8 -> 75.2 ms;
// Philox inlined again with those: 82.1 ms; a single Philox call site per sampler: 76.7 ms (profiles/r2_52, r2_53).
// ------------------------------------------------------------------ Philox-4x32-10 / PathRng
RT_DEV uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        if (r) { k.x += 0x9E3779B9u; k.y += 0xBB67AE85u; }
        const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    }
    return c;
}
// One out-of-line copy for the fused kernels, whose ~19 inlined call sites cost 8 KB of code (see the A/B note above)
static __device__ __noinline__ uint4 philox4x32_10_ool(uint4 c, uint2 k) { return philox4x32_10(c, k); }

// Draw k of a path = word (k & 3) of block (path_lo, path_hi, k >> 2, 0) under key (seed_lo, seed_hi);
// xi = u32 * 2^-32 (SURVEY.md Appendix D; identical in oracle/rt_oracle.hpp PathCtx); scatters start on block boundaries.
template <bool OOL>
struct PathRngT {
    RT_DEV uint4 block(uint32_t b) const {
        const uint4 c = make_uint4(path.x, path.y, b, 0u);
        return OOL ? philox4x32_10_ool(c, key) : philox4x32_10(c, key);
    }
    uint2 key, path;
    uint32_t draw, cached; // cached = index of the block held in blk
    uint4 blk;
    RT_DEV void init(uint64_t seed, uint64_t path_id, uint32_t draw0) {
        key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
        path = make_uint2((uint32_t)path_id, (uint32_t)(path_id >> 32));
        draw = draw0;
        cached = 0xffffffffu;
    }
    // RNG contract: every Material::scatter starts at the next multiple-of-4 draw index (as PathCtx::begin_event
    // in the oracle).  The first block of the event is generated right here, while all lanes of the material
    // branch are still together, instead of inside the diverged rejection loop.
    RT_DEV void begin_event() {
        draw = (draw + 3u) & ~3u;
        const uint32_t b = draw >> 2;
        blk = block(b);
        cached = b;
    }
    RT_DEV uint32_t next_u32() {
        const uint32_t b = draw >> 2;
        if (b != cached) {
            blk = block(b);
            cached = b;
        }
        const uint32_t w = draw & 3u;
        ++draw;
        return w == 0 ? blk.x : (w == 1 ? blk.y : (w == 2 ? blk.z : blk.w));
    }
    // xi = u * 2^-32 and 2 xi - 1 without an integer -> double conversion: the bits (0x43300000, u) ARE the double 2^52 + u, and
    // (2^52 + u) * 2^-32 - 2^20 = u * 2^-32, (2^52 + u) * 2^-31 - (2^21 + 1) = u * 2^-31 - 1 are exact, so one fma returns the very
    // double that (double)u * 2^-32 resp. fma(xi, 2.0, -1.0) round to (they are exact as well)
    static RT_DEV double unit_of(uint32_t u) { return fma(__hiloint2double(0x43300000, (int)u), 1.0 / 4294967296.0, -1048576.0); }
    static RT_DEV double pm1_of(uint32_t u) { return fma(__hiloint2double(0x43300000, (int)u), 1.0 / 2147483648.0, -2097153.0); }
    RT_DEV double gen() { return unit_of(next_u32()); }
    RT_DEV double gen_range(double a, double b) { return fma(gen(), b - a, a); }
    // The next two / three draws as gen_range(-1, 1) values, for the rejection samplers (random_in_unit_sphere, random_in_unit_disk):
    // the same words of the same blocks as two / three next_u32() calls, picked with selects instead of a branch ladder per draw
    // (the loops run at 5-6 of 32 lanes and were a quarter of the fused kernels' instructions, profiles/README.md)
    RT_DEV void next3_pm1(double& a, double& b, double& c) {
        const uint32_t bi = draw >> 2, w = draw & 3u;
        if (bi != cached) { blk = block(bi); cached = bi; }
        uint4 nb = blk;
        if (w >= 2u) nb = block(bi + 1u);
        const bool w1 = (w & 1u) != 0, w2 = (w & 2u) != 0;
        a = pm1_of(w2 ? (w1 ? blk.w : blk.z) : (w1 ? blk.y : blk.x));
        b = pm1_of(w2 ? (w1 ? nb.x : blk.w) : (w1 ? blk.z : blk.y));
        c = pm1_of(w2 ? (w1 ? nb.y : nb.x) : (w1 ? blk.w : blk.z));
        if (w >= 2u) { blk = nb; cached = bi + 1u; }
        draw += 3u;
    }
    RT_DEV void next2_pm1(double& a, double& b) {
        const uint32_t bi = draw >> 2, w = draw & 3u;
        if (bi != cached) { blk = block(bi); cached = bi; }
        uint4 nb = blk;
        if (w == 3u) nb = block(bi + 1u);
        const bool w1 = (w & 1u) != 0, w2 = (w & 2u) != 0;
        a = pm1_of(w2 ? (w1 ? blk.w : blk.z) : (w1 ? blk.y : blk.x));
        b = pm1_of(w2 ? (w1 ? nb.x : blk.w) : (w1 ? blk.z : blk.y));
        if (w == 3u) { blk = nb; cached = bi + 1u; }
        draw += 2u;
    }
};
using PathRng = PathRngT<false>;    // wavefront kernels, parity hooks
using PathRngOol = PathRngT<true>;  // fused kernels
// The fused kernels open the event ONCE for all lanes that scatter, before the branch on the material type, and hand the samplers
// this type, whose own begin_event() does nothing: one Philox call at ~20 lanes instead of one per material present in the warp
struct PathRngOolBegun : PathRngOol {
    RT_DEV void open_event() { PathRngOol::begin_event(); }
    RT_DEV void begin_event() {}
};
RT_DEV double medium_xi(uint64_t seed, uint64_t path_id, uint32_t medium_prim_id, uint32_t segment) {
    const uint4 o = philox4x32_10(make_uint4((uint32_t)path_id, (uint32_t)(path_id >> 32), medium_prim_id, 0x80000000u | segment),
                                  make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    return (double)o.x * (1.0 / 4294967296.0);
}

template <class G> RT_DEV D3 random_in_unit_sphere(G& g) { // vec3.rs:287-295
    for (;;) {
        double a, b, c;
        g.next3_pm1(a, b, c);
        const D3 p = mk3(a, b, c);
        if (length_squared(p) < 1.0) return p;
    }
}
template <class G> RT_DEV D3 random_unit_vector(G& g) { return unit(random_in_unit_sphere(g)); } // vec3.rs:297-299

// ------------------------------------------------------------------ transforms (hit.rs:802-807, 893-904)
RT_DEV void xform_ray(const XformOp* __restrict__ ops, uint32_t off, uint32_t len, Ray& r) {
    for (uint32_t i = 0; i < len; ++i) {
        const XformOp op = ops[off + i];
        if (op.type == XF_TRANSLATE) {
            r.o = mk3(r.o.x - op.a, r.o.y - op.b, r.o.z - op.c);
        } else {
            const double s = op.a, c = op.b;
            r.o = mk3(c * r.o.x - s * r.o.z, r.o.y, s * r.o.x + c * r.o.z);
            r.d = mk3(c * r.d.x - s * r.d.z, r.d.y, s * r.d.x + c * r.d.z);
        }
    }
}

// ------------------------------------------------------------------ best-hit bookkeeping
struct BestHit {
    double t;      // closest_so_far
    uint32_t type; // PrimType, 0xffffffff = nothing found yet
    uint32_t idx, side, inst;
};
#define RT_NONE 0xffffffffu
#define RT_INF (__longlong_as_double(0x7ff0000000000000LL))
RT_DEV void best_init(BestHit& b, double t_max) { b.t = t_max; b.type = RT_NONE; b.idx = 0; b.side = 0; b.inst = 0; }

// Accepts t <= closest_so_far like the reference's list scan (hit.rs:675-683: the later element wins
// an exact tie).  Ties are decided by the depth-first leaf id, fetched only when a tie happens.
RT_DEV void consider(const DeviceScene& S, BestHit& best, double t, uint32_t type, uint32_t idx, uint32_t side, uint32_t inst) {
    bool ok = (t <= best.t) & (t < RT_INF); // NaN and +inf are rejected (documented divergence: the reference lets t = +inf through)
    if (ok & (t == best.t) & (best.type != RT_NONE)) { // the one (rare) branch; the update below is selects (see box_side_ok)
        const uint32_t pid_new = __ldg(&S.meta[type][idx].prim_id) + side;
        const uint32_t pid_old = __ldg(&S.meta[best.type][best.idx].prim_id) + best.side;
        ok = !(pid_new < pid_old);
    }
    best.t = ok ? t : best.t; best.type = ok ? type : best.type; best.idx = ok ? idx : best.idx; best.side = ok ? side : best.side;
    best.inst = ok ? inst : best.inst;
}

// ------------------------------------------------------------------ primitive tests (f64)
// Sphere / MovingSphere / GravitySphere::hit root selection (hit.rs:204-222, 282-300, 398-416).
// a = d.d and 1/a depend only on the ray: computed once per ray per instance (RayPre).
struct RayPre {
    double a, inv_a;
    D3 inv_d; // 1 / direction per axis, for the axis-aligned plane tests (rects, box sides)
};
RT_DEV RayPre make_raypre(const Ray& r, bool planar) {
    RayPre p;
    p.a = length_squared(r.d);
    p.inv_a = 1.0 / p.a;
    p.inv_d = mk3(0, 0, 0);
    if (planar) p.inv_d = mk3(1.0 / r.d.x, 1.0 / r.d.y, 1.0 / r.d.z);
    return p;
}
RT_DEV double sphere_root(const Ray& r, const RayPre& pre, D3 c, double radius, double t_min, double t_max) {
    const D3 oc = r.o - c;
    const double half_b = dot(oc, r.d);
    const double cc = fma(-radius, radius, length_squared(oc));
    const double disc = fma(half_b, half_b, -(pre.a * cc));
    if (disc < 0.0) return RT_INF;
    const double sqrtd = sqrt(disc);
    double root = (-half_b - sqrtd) * pre.inv_a;
    if (root < t_min || t_max < root) {
        root = (-half_b + sqrtd) * pre.inv_a;
        if (root < t_min || t_max < root) return RT_INF;
    }
    return root;
}
RT_DEV D3 moving_center(const DMoving& m, double time) { // hit.rs:275-278
    const double f = (time - m.t0) / m.dt;
    return mk3(fma(f, m.dc[0], m.c0[0]), fma(f, m.dc[1], m.c0[1]), fma(f, m.dc[2], m.c0[2]));
}
RT_DEV D3 gravity_center(const DeviceScene& S, const DGravity& g, double time) { // hit.rs:370-379
    const double q = time / 0.001;
    int64_t i = (q > 0.0) ? (int64_t)q : 0; // Rust `as usize`: saturating, negative/NaN -> 0
    i -= g.idx0;
    i = i < 0 ? 0 : (i >= g.n ? g.n - 1 : i); // window uploaded for the camera shutter; clamped
    return mk3(g.x, __ldg(&S.gravity_table[g.table_off + (int32_t)i]), g.z);
}
// XyRect / XzRect / YzRect::hit (hit.rs:476-485, 541-550, 606-615): returns t or +inf.
// t = (k - o) / d is evaluated as (k - o) * (1/d) with the per-ray reciprocal (<= 1 ulp from the division).
RT_DEV double rect_t(const Ray& r, const RayPre& pre, const DRect& q, double t_min, double t_max) {
    const int ax = q.axis;
    const int ia = ax == 0 ? 1 : 0, ib = ax == 2 ? 1 : 2;
    const double t = (q.k - axis_of(r.o, ax)) * axis_of(pre.inv_d, ax);
    if (t < t_min || t > t_max) return RT_INF;
    const double x = fma(t, axis_of(r.d, ia), axis_of(r.o, ia));
    const double y = fma(t, axis_of(r.d, ib), axis_of(r.o, ib));
    if (x < q.a0 || x > q.a1 || y < q.b0 || y > q.b1) return RT_INF;
    return t;
}
// One side of a RectPrism (hit.rs:722-769): s = 0..5 -> +z(p1.z), -z(p0.z), +y, -y, +x, -x.  Returns t or +inf.
RT_DEV double box_side_t(const Ray& r, const RayPre& pre, const DBox& b, int s) {
    const int ax = s < 2 ? 2 : (s < 4 ? 1 : 0);
    const int ia = ax == 0 ? 1 : 0, ib = ax == 2 ? 1 : 2;
    const double k = (s & 1) ? b.p0[ax] : b.p1[ax];
    const double t = (k - axis_of(r.o, ax)) * axis_of(pre.inv_d, ax);
    if (!(t < RT_INF) || !(t > -RT_INF)) return RT_INF;
    const double x = fma(t, axis_of(r.d, ia), axis_of(r.o, ia));
    const double y = fma(t, axis_of(r.d, ib), axis_of(r.o, ib));
    if (x < b.p0[ia] || x > b.p1[ia] || y < b.p0[ib] || y > b.p1[ib]) return RT_INF;
    return t;
}
// RectPrism = HittableList of six rects scanned in order with a shrinking closest_so_far
// (hit.rs:660-690).  Returns t and the winning side (later side wins an exact tie).
// Branch-free form of one side: the same t, the same hit point and the same comparisons as box_side_t + the scan's own tests, folded
// into one predicate (a side whose t is not finite, or that misses the rect, or that lies outside [t_min, closest] changes nothing).
// Round 2: early returns are what costs in the leaf code, which runs at 2-8 of 32 lanes (branch / reconvergence / instruction-fetch
// stalls per useful instruction): box sides book-2 final +6.2 %, Cornell smoke +1.3 %; consider() 871 200-triangle mesh +3.0 %;
// triangle test mesh +2.5 %; the same treatment LOSES on sphere_root (book-1 final -3 %) and is neutral on rect_t, which keep their
// early returns (profiles/r2_61 ... r2_64).
RT_DEV bool box_side_ok(const Ray& r, const RayPre& pre, const DBox& b, int s, double t_min, double closest, double& t) {
    const int ax = s < 2 ? 2 : (s < 4 ? 1 : 0);
    const int ia = ax == 0 ? 1 : 0, ib = ax == 2 ? 1 : 2;
    const double k = (s & 1) ? b.p0[ax] : b.p1[ax];
    t = (k - axis_of(r.o, ax)) * axis_of(pre.inv_d, ax);
    const double x = fma(t, axis_of(r.d, ia), axis_of(r.o, ia));
    const double y = fma(t, axis_of(r.d, ib), axis_of(r.o, ib));
    return (t < RT_INF) & (t > -RT_INF) & !(x < b.p0[ia]) & !(x > b.p1[ia]) & !(y < b.p0[ib]) & !(y > b.p1[ib]) & !(t < t_min) & !(t > closest);
}
RT_DEV double box_t(const Ray& r, const RayPre& pre, const DBox& b, double t_min, double t_max, uint32_t& side_out) {
    double closest = t_max;
    bool any = false;
    uint32_t side = 0;
#pragma unroll
    for (int s = 0; s < 6; ++s) {
        double t;
        const bool ok = box_side_ok(r, pre, b, s, t_min, closest, t);
        closest = ok ? t : closest; side = ok ? (uint32_t)s : side; any = any | ok;
    }
    side_out = side;
    return any ? closest : RT_INF;
}
// Triangle::hit (hit.rs:111-149): plane hit + three inclusive edge tests; vertices/normal stored f32
RT_DEV double tri_t(const Ray& r, const DTri* __restrict__ tp, double t_min, double t_max) {
    const float4 q0 = __ldg(reinterpret_cast<const float4*>(tp));
    const float4 q1 = __ldg(reinterpret_cast<const float4*>(tp) + 1);
    const float4 q2 = __ldg(reinterpret_cast<const float4*>(tp) + 2);
    const D3 v0 = mk3(q0.x, q0.y, q0.z), v1 = mk3(q0.w, q1.x, q1.y), v2 = mk3(q1.z, q1.w, q2.x), n = mk3(q2.y, q2.z, q2.w);
    const double nd = dot(n, r.d);
    const double dd = __ldg(&tp->dd); // -(n . v0) with the exact f64 vertex (rt_types.h DTri)
    // the reference's five tests (|n.d| cutoff, t range, three inclusive edge tests) as one predicate instead of five early returns:
    // a rejected t still yields a point whose edge tests are ignored (see box_side_ok)
    const double t = -(dot(n, r.o) + dd) / nd;
    const D3 p = ray_at(r, t);
    const bool miss = (fabs(nd) < 0.0001) | (t < t_min) | (t > t_max) | (dot(n, cross(v1 - v0, p - v0)) < 0.0) | (dot(n, cross(v2 - v1, p - v1)) < 0.0) |
                      (dot(n, cross(v0 - v2, p - v2)) < 0.0);
    return miss ? RT_INF : t;
}

// ------------------------------------------------------------------ BVH traversal (aabb.rs:23-61, bvh.rs:97-112)
struct RayF {
    float idx, idy, idz, oodx, oody, oodz;
};
RT_DEV RayF make_rayf(const Ray& r) {
    RayF f;
    float dx = (float)r.d.x, dy = (float)r.d.y, dz = (float)r.d.z;
    const float tiny = 1e-20f; // exact zeros become +-tiny so that no slab distance is inf - inf
    dx = fabsf(dx) < tiny ? copysignf(tiny, dx) : dx;
    dy = fabsf(dy) < tiny ? copysignf(tiny, dy) : dy;
    dz = fabsf(dz) < tiny ? copysignf(tiny, dz) : dz;
    f.idx = 1.0f / dx; f.idy = 1.0f / dy; f.idz = 1.0f / dz;
    f.oodx = (float)r.o.x * f.idx; f.oody = (float)r.o.y * f.idy; f.oodz = (float)r.o.z * f.idz;
    return f;
}
RT_DEV bool slab(const float4 lo, const float4 hi, const RayF& f, float t_min, float t_max, float& tn) {
    const float x0 = fmaf(lo.x, f.idx, -f.oodx), x1 = fmaf(hi.x, f.idx, -f.oodx);
    const float y0 = fmaf(lo.y, f.idy, -f.oody), y1 = fmaf(hi.y, f.idy, -f.oody);
    const float z0 = fmaf(lo.z, f.idz, -f.oodz), z1 = fmaf(hi.z, f.idz, -f.oodz);
    tn = fmaxf(fmaxf(fminf(x0, x1), fminf(y0, y1)), fmaxf(fminf(z0, z1), t_min));
    const float tf = fminf(fminf(fmaxf(x0, x1), fmaxf(y0, y1)), fminf(fmaxf(z0, z1), t_max));
    return tn <= tf;
}
RT_DEV float f32_up(double v) { return __double2float_ru(v); }
RT_DEV float f32_down(double v) { return __double2float_rd(v); }

struct TraceCounters {
    uint32_t nodes, prims;
};

// PM = compile-time mask of the primitive types the scene can contain (bit = PrimType): kernels specialised
// for "spheres only" etc. drop the other tests from the hot loop.
#define RT_PM_ALL 0x3fu
#define RT_PM_HAS(PM, T) (((PM) >> (T)) & 1u)
#define RT_PAIR_BOUND(PM) (((PM) == 0x3u || (PM) == 0x5u) ? 2 : 0) // node steps of the sibling-pair walk before pending leaves are tested; 0 = unbounded
// Tests every primitive of one leaf against the object-space ray.
template <uint32_t PM = RT_PM_ALL>
RT_DEV void leaf_test(const DeviceScene& S, const Ray& r, const RayPre& pre, double t_min, BestHit& best, uint32_t type, uint32_t first, uint32_t n,
                      uint32_t inst) {
    for (uint32_t i = first; i < first + n; ++i) {
        if ((PM & 7u) && ((PM & ~7u) == 0 || type <= PRIM_GRAVITY)) { // the three sphere kinds share the root solve (hit.rs:204-222, 282-300, 398-416)
            D3 c;
            double rad;
            if (RT_PM_HAS(PM, PRIM_SPHERE) && ((PM & 6u) == 0 || type == PRIM_SPHERE)) {
                const double2 a = __ldg(reinterpret_cast<const double2*>(&S.spheres[i]));
                const double2 b = __ldg(reinterpret_cast<const double2*>(&S.spheres[i]) + 1);
                c = mk3(a.x, a.y, b.x); rad = b.y;
            } else if (RT_PM_HAS(PM, PRIM_MOVING) && (!RT_PM_HAS(PM, PRIM_GRAVITY) || type == PRIM_MOVING)) {
                const DMoving m = S.movings[i];
                c = moving_center(m, r.time); rad = m.r;
            } else {
                const DGravity g = S.gravities[i];
                c = gravity_center(S, g, r.time); rad = g.r;
            }
            consider(S, best, sphere_root(r, pre, c, rad, t_min, best.t), type, i, 0, inst);
        } else if (RT_PM_HAS(PM, PRIM_RECT) && type == PRIM_RECT) {
            const DRect q = S.rects[i];
            consider(S, best, rect_t(r, pre, q, t_min, best.t), type, i, 0, inst);
        } else if (RT_PM_HAS(PM, PRIM_BOX) && type == PRIM_BOX) {
            const DBox b = S.boxes[i];
            uint32_t side;
            const double t = box_t(r, pre, b, t_min, best.t, side);
            consider(S, best, t, type, i, side, inst);
        } else if (RT_PM_HAS(PM, PRIM_TRI)) { // PRIM_TRI
            consider(S, best, tri_t(r, &S.tris[i], t_min, best.t), type, i, 0, inst);
        }
    }
}

// Closest hit inside one instance; `r` is already in the instance's space.
//
// "while-while" traversal: each lane walks interior nodes until it holds a pending leaf (or is done);
// only when every lane of the warp has left that inner loop are the leaves processed, so the expensive
// f64 primitive tests run with as many lanes active as possible.  The instance root is stored as the
// first node of a sibling pair whose second node is an empty leaf, so the root needs no special case.
// Speculative while-while (Aila & Laine): a lane that holds one pending leaf keeps walking until it has a second one (or
// runs out of nodes), so fewer lanes idle in the node loop; up to three leaves are then tested together.  Measured
// (tools/ab_libs.sh): Cornell smoke +3.7 %, book-1 +0.4 %, book-2 final -8.5 % (its speculative walks test more boxes of
// the 400-box floor): used by the rects + boxes kernels only.
template <bool COUNT, uint32_t PM = RT_PM_ALL>
RT_DEV void trace_instance_spec(const DeviceScene& S, uint32_t inst_idx, const Ray& r, double t_min, BestHit& best, TraceCounters* cnt) {
    const RayF f = make_rayf(r);
    const RayPre pre = make_raypre(r, (PM & 0x18u) != 0 && (S.flags & 1u) != 0);
    const float tminf = f32_down(t_min);
    float tmaxf = f32_up(best.t);
    const float4* __restrict__ nodes = reinterpret_cast<const float4*>(S.nodes);
    uint32_t stack[RT_STACK];
    int sp = 0;
    const uint32_t DONE = 0xffffffffu;
    uint32_t cur = __ldg(&S.instances[inst_idx].root);
    while (cur != DONE) {
        uint32_t lf0 = 0, lc0 = 0, lf1 = 0, lc1 = 0, lf2 = 0, lc2 = 0;
        while (cur != DONE && lc1 == 0) { // at most one leaf pending: a pair can add two
            const float4 lo0 = __ldg(nodes + 2 * cur), hi0 = __ldg(nodes + 2 * cur + 1);
            const float4 lo1 = __ldg(nodes + 2 * cur + 2), hi1 = __ldg(nodes + 2 * cur + 3);
            float tn0, tn1;
            bool h0 = slab(lo0, hi0, f, tminf, tmaxf, tn0);
            bool h1 = slab(lo1, hi1, f, tminf, tmaxf, tn1);
            if (COUNT) cnt->nodes += 2;
            const uint32_t c0 = __float_as_uint(hi0.w), c1 = __float_as_uint(hi1.w);
            if (h0 && c0) {
                const uint32_t a = __float_as_uint(lo0.w), b = c0 & 0x7fffffffu;
                if (lc0 == 0) { lf0 = a; lc0 = b; } else { lf1 = a; lc1 = b; }
                h0 = false;
            }
            if (h1 && c1) {
                const uint32_t a = __float_as_uint(lo1.w), b = c1 & 0x7fffffffu;
                if (lc0 == 0) { lf0 = a; lc0 = b; } else if (lc1 == 0) { lf1 = a; lc1 = b; } else { lf2 = a; lc2 = b; }
                h1 = false;
            }
            if (h0 && h1) {
                const uint32_t n0 = __float_as_uint(lo0.w), n1 = __float_as_uint(lo1.w);
                const bool first0 = tn0 <= tn1;
                cur = first0 ? n0 : n1;
                if (sp < RT_STACK) stack[sp++] = first0 ? n1 : n0;
            } else if (h0) {
                cur = __float_as_uint(lo0.w);
            } else if (h1) {
                cur = __float_as_uint(lo1.w);
            } else {
                cur = sp ? stack[--sp] : DONE;
            }
        }
        for (int k = 0; k < 3; ++k) { // runtime loop: one copy of the primitive code
            const uint32_t lc = k == 0 ? lc0 : (k == 1 ? lc1 : lc2), lf = k == 0 ? lf0 : (k == 1 ? lf1 : lf2);
            if (lc & 0xffffffu) {
                if (COUNT) cnt->prims += lc & 0xffffffu;
                leaf_test<PM>(S, r, pre, t_min, best, lc >> 24, lf, lc & 0xffffffu, inst_idx);
            }
        }
        tmaxf = f32_up(best.t);
    }
}

template <bool COUNT, uint32_t PM = RT_PM_ALL>
RT_DEV void trace_instance(const DeviceScene& S, uint32_t inst_idx, const Ray& r, double t_min, BestHit& best, TraceCounters* cnt) {
    const RayF f = make_rayf(r);
    const RayPre pre = make_raypre(r, (PM & 0x18u) != 0 && (S.flags & 1u) != 0);
    const float tminf = f32_down(t_min);
    float tmaxf = f32_up(best.t);
    const float4* __restrict__ nodes = reinterpret_cast<const float4*>(S.nodes);
    // the spheres + moving-spheres kernels walk motion-interpolated boxes (DeviceScene::mnodes) when the scene has them
    const float4* __restrict__ mnodes = reinterpret_cast<const float4*>(S.mnodes);
    const bool MOTION = PM == 0x3u && mnodes != nullptr;
    float ms = 0.f;
    if (MOTION) { const double sd = (r.time - S.motion_t0) * S.motion_inv_dt; ms = (float)(sd < 0.0 ? 0.0 : (sd > 1.0 ? 1.0 : sd)); }
    uint32_t stack[RT_STACK];
    int sp = 0;
    const uint32_t DONE = 0xffffffffu;
    uint32_t cur = __ldg(&S.instances[inst_idx].root);
    while (cur != DONE) {
        uint32_t leaf_first0 = 0, leaf_cnt0 = 0, leaf_first1 = 0, leaf_cnt1 = 0; // cnt = (type << 24) | n, 0 = none
        // bounded node loop for the spheres + moving / gravity spheres kernels (see walk_wide): 2 steps, then the pending leaves are looked at
        // (book-1 as shipped 169.0 -> 156.6 ms per 500 spp); unbounded elsewhere (Cornell smoke and book-2 final lose 2-9 % with any bound)
        int inner = 0;
#pragma unroll 1
        while (cur != DONE && (leaf_cnt0 | leaf_cnt1) == 0 && (RT_PAIR_BOUND(PM) == 0 || inner++ < RT_PAIR_BOUND(PM))) {
            // cur = index of the left node of a sibling pair: one 64-byte fetch, two slab tests
            float4 lo0, hi0, lo1, hi1;
            if (MOTION) { // box(t) = box at the shutter's start + s * delta: 128 bytes per sibling pair
                lo0 = __ldg(mnodes + 4 * cur); hi0 = __ldg(mnodes + 4 * cur + 1);
                lo1 = __ldg(mnodes + 4 * cur + 4); hi1 = __ldg(mnodes + 4 * cur + 5);
                const float4 dl0 = __ldg(mnodes + 4 * cur + 2), dh0 = __ldg(mnodes + 4 * cur + 3);
                const float4 dl1 = __ldg(mnodes + 4 * cur + 6), dh1 = __ldg(mnodes + 4 * cur + 7);
                lo0.x = fmaf(dl0.x, ms, lo0.x); lo0.y = fmaf(dl0.y, ms, lo0.y); lo0.z = fmaf(dl0.z, ms, lo0.z);
                hi0.x = fmaf(dh0.x, ms, hi0.x); hi0.y = fmaf(dh0.y, ms, hi0.y); hi0.z = fmaf(dh0.z, ms, hi0.z);
                lo1.x = fmaf(dl1.x, ms, lo1.x); lo1.y = fmaf(dl1.y, ms, lo1.y); lo1.z = fmaf(dl1.z, ms, lo1.z);
                hi1.x = fmaf(dh1.x, ms, hi1.x); hi1.y = fmaf(dh1.y, ms, hi1.y); hi1.z = fmaf(dh1.z, ms, hi1.z);
            } else {
                lo0 = __ldg(nodes + 2 * cur); hi0 = __ldg(nodes + 2 * cur + 1);
                lo1 = __ldg(nodes + 2 * cur + 2); hi1 = __ldg(nodes + 2 * cur + 3);
            }
            float tn0, tn1;
            bool h0 = slab(lo0, hi0, f, tminf, tmaxf, tn0);
            bool h1 = slab(lo1, hi1, f, tminf, tmaxf, tn1);
            if (COUNT) cnt->nodes += 2;
            const uint32_t c0 = __float_as_uint(hi0.w), c1 = __float_as_uint(hi1.w);
            if (h0 && c0) { leaf_first0 = __float_as_uint(lo0.w); leaf_cnt0 = c0 & 0x7fffffffu; h0 = false; }
            if (h1 && c1) { leaf_first1 = __float_as_uint(lo1.w); leaf_cnt1 = c1 & 0x7fffffffu; h1 = false; }
            if (h0 && h1) {
                const uint32_t n0 = __float_as_uint(lo0.w), n1 = __float_as_uint(lo1.w);
                const bool first0 = tn0 <= tn1;
                cur = first0 ? n0 : n1;
                if (sp < RT_STACK) stack[sp++] = first0 ? n1 : n0;
            } else if (h0) {
                cur = __float_as_uint(lo0.w);
            } else if (h1) {
                cur = __float_as_uint(lo1.w);
            } else {
                cur = sp ? stack[--sp] : DONE;
            }
        }
        for (int k = 0; k < 2; ++k) { // runtime loop: one copy of the primitive code
            const uint32_t lc = k ? leaf_cnt1 : leaf_cnt0, lf = k ? leaf_first1 : leaf_first0;
            if (lc & 0xffffffu) {
                if (COUNT) cnt->prims += lc & 0xffffffu;
                leaf_test<PM>(S, r, pre, t_min, best, lc >> 24, lf, lc & 0xffffffu, inst_idx);
            }
        }
        tmaxf = f32_up(best.t);
    }
}

// Resumable form of trace_instance for the fused kernel (single instance, no wrappers).  The walk is the
// same; its state (cur, sp, stack, best) lives in the caller, and the warp leaves the loop as soon as
// `wait_thresh` of the lanes that entered with work have finished, instead of idling them until the slowest
// lane is done.  The unfinished lanes come back with the next call (after the finished ones have shaded and
// started their next segment) and continue where they stopped.  Called by all 32 lanes.
// walk_pairs = the loop of trace_resume with the per-ray constants (f32 reciprocals, a = d.d, 1/a, 1/d) supplied by the caller, who keeps
// them in registers across calls (k_pool: a lane's walk is suspended and resumed many times), and with the lane's instance index for
// the hit record.  MOTION: spheres + moving spheres scenes walk the motion-interpolated boxes (DeviceScene::mnodes) like trace_instance.
template <uint32_t PM = RT_PM_ALL>
RT_DEV void walk_pairs(const DeviceScene& S, const Ray& r, const RayF& f, const RayPre& pre, double t_min, BestHit& best, uint32_t& cur, int& sp, uint32_t* stack,
                       uint32_t wait_thresh, uint32_t inst) {
    const unsigned full = 0xffffffffu;
    const float tminf = f32_down(t_min);
    float tmaxf = f32_up(best.t);
    const float4* __restrict__ nodes = reinterpret_cast<const float4*>(S.nodes);
    const float4* __restrict__ mnodes = reinterpret_cast<const float4*>(S.mnodes);
    const bool MOTION = PM == 0x3u && mnodes != nullptr;
    float ms = 0.f;
    if (MOTION) { const double sd = (r.time - S.motion_t0) * S.motion_inv_dt; ms = (float)(sd < 0.0 ? 0.0 : (sd > 1.0 ? 1.0 : sd)); }
    const uint32_t DONE = 0xffffffffu;
    const uint32_t n0 = __popc(__ballot_sync(full, cur != DONE));
    for (;;) {
        uint32_t leaf_first0 = 0, leaf_cnt0 = 0, leaf_first1 = 0, leaf_cnt1 = 0;
        // bounded node loop for the spheres + moving / gravity spheres kernels (see walk_wide): 2 steps, then the pending leaves are looked at
        // (book-1 as shipped 169.0 -> 156.6 ms per 500 spp); unbounded elsewhere (Cornell smoke and book-2 final lose 2-9 % with any bound)
        int inner = 0;
#pragma unroll 1
        while (cur != DONE && (leaf_cnt0 | leaf_cnt1) == 0 && (RT_PAIR_BOUND(PM) == 0 || inner++ < RT_PAIR_BOUND(PM))) {
            float4 lo0, hi0, lo1, hi1;
            if (MOTION) {
                lo0 = __ldg(mnodes + 4 * cur); hi0 = __ldg(mnodes + 4 * cur + 1);
                lo1 = __ldg(mnodes + 4 * cur + 4); hi1 = __ldg(mnodes + 4 * cur + 5);
                const float4 dl0 = __ldg(mnodes + 4 * cur + 2), dh0 = __ldg(mnodes + 4 * cur + 3);
                const float4 dl1 = __ldg(mnodes + 4 * cur + 6), dh1 = __ldg(mnodes + 4 * cur + 7);
                lo0.x = fmaf(dl0.x, ms, lo0.x); lo0.y = fmaf(dl0.y, ms, lo0.y); lo0.z = fmaf(dl0.z, ms, lo0.z);
                hi0.x = fmaf(dh0.x, ms, hi0.x); hi0.y = fmaf(dh0.y, ms, hi0.y); hi0.z = fmaf(dh0.z, ms, hi0.z);
                lo1.x = fmaf(dl1.x, ms, lo1.x); lo1.y = fmaf(dl1.y, ms, lo1.y); lo1.z = fmaf(dl1.z, ms, lo1.z);
                hi1.x = fmaf(dh1.x, ms, hi1.x); hi1.y = fmaf(dh1.y, ms, hi1.y); hi1.z = fmaf(dh1.z, ms, hi1.z);
            } else {
                lo0 = __ldg(nodes + 2 * cur); hi0 = __ldg(nodes + 2 * cur + 1);
                lo1 = __ldg(nodes + 2 * cur + 2); hi1 = __ldg(nodes + 2 * cur + 3);
            }
            float tn0, tn1;
            bool h0 = slab(lo0, hi0, f, tminf, tmaxf, tn0);
            bool h1 = slab(lo1, hi1, f, tminf, tmaxf, tn1);
            const uint32_t c0 = __float_as_uint(hi0.w), c1 = __float_as_uint(hi1.w);
            if (h0 && c0) { leaf_first0 = __float_as_uint(lo0.w); leaf_cnt0 = c0 & 0x7fffffffu; h0 = false; }
            if (h1 && c1) { leaf_first1 = __float_as_uint(lo1.w); leaf_cnt1 = c1 & 0x7fffffffu; h1 = false; }
            if (h0 && h1) {
                const uint32_t n0i = __float_as_uint(lo0.w), n1i = __float_as_uint(lo1.w);
                const bool first0 = tn0 <= tn1;
                cur = first0 ? n0i : n1i;
                if (sp < RT_STACK) stack[sp++] = first0 ? n1i : n0i;
            } else if (h0) {
                cur = __float_as_uint(lo0.w);
            } else if (h1) {
                cur = __float_as_uint(lo1.w);
            } else {
                cur = sp ? stack[--sp] : DONE;
            }
        }
        for (int k = 0; k < 2; ++k) {
            const uint32_t lc = k ? leaf_cnt1 : leaf_cnt0, lf = k ? leaf_first1 : leaf_first0;
            if (lc & 0xffffffu) leaf_test<PM>(S, r, pre, t_min, best, lc >> 24, lf, lc & 0xffffffu, inst);
        }
        tmaxf = f32_up(best.t);
        const uint32_t still = __popc(__ballot_sync(full, cur != DONE));
        if (still == 0 || n0 - still >= wait_thresh) break;
    }
}

template <uint32_t PM = RT_PM_ALL>
RT_DEV void trace_resume(const DeviceScene& S, const Ray& r, double t_min, BestHit& best, uint32_t& cur, int& sp, uint32_t* stack, uint32_t wait_thresh) {
    const RayF f = make_rayf(r);
    const RayPre pre = make_raypre(r, (PM & 0x18u) != 0 && (S.flags & 1u) != 0);
    walk_pairs<PM>(S, r, f, pre, t_min, best, cur, sp, stack, wait_thresh, 0u);
}

// ------------------------------------------------------------------ 4-wide walk (rt_types.h RT_WIDE_EMPTY, host/bvh_wide.hpp)
// One 128-byte node = four child boxes in SoA form + four references.  The children that the ray's interval reaches are
// keyed by entry distance (64-bit keys = distance bits << 32 | reference); three compare-exchanges find the nearest, which becomes
// `cur`, the others are pushed.  Leaves travel through the stack like nodes, and an entry whose entry distance
// has fallen behind closest_so_far is dropped when popped, so no primitive of a box that a nearer hit already culled is
// tested.  Same closest hit as the binary walk (topology independent; ties by depth-first id in consider()).
// Requires t_min >= 0 (distance bits are compared as unsigned integers).
#ifndef RT_WIDE_SIGNED
#define RT_WIDE_SIGNED 1 // 0 = the per-box min / max form (A/B: book-1 final 83.5 -> 80.8 ms, mesh +1.8 % with 1)
#endif
RT_DEV unsigned long long wide_key(float lx, float hx, float ly, float hy, float lz, float hz, float ref, const RayF& f, float t_min, float t_max) {
    const float x0 = fmaf(lx, f.idx, -f.oodx), x1 = fmaf(hx, f.idx, -f.oodx);
    const float y0 = fmaf(ly, f.idy, -f.oody), y1 = fmaf(hy, f.idy, -f.oody);
    const float z0 = fmaf(lz, f.idz, -f.oodz), z1 = fmaf(hz, f.idz, -f.oodz);
    const float tn = fmaxf(fmaxf(fminf(x0, x1), fminf(y0, y1)), fmaxf(fminf(z0, z1), t_min));
    const float tf = fminf(fminf(fmaxf(x0, x1), fmaxf(y0, y1)), fminf(fmaxf(z0, z1), t_max));
    const uint32_t r = __float_as_uint(ref);
    if (!(tn <= tf) || r == RT_WIDE_EMPTY) return ~0ull;
    return ((unsigned long long)(__float_as_uint(tn) & 0x7fffffffu) << 32) | (unsigned long long)r;
}
// The same key from the planes the ray enters / leaves through, picked per RAY (by the sign of 1/d) when the node rows are loaded
// instead of per box with six min / max: 1/d is finite and non-zero (make_rayf) and lo <= hi, so fma(lo, idx, -ood) <= fma(hi, idx, -ood)
// for idx > 0 and >= for idx < 0 (a correctly rounded fma is monotonic): min(x0, x1) and max(x0, x1) ARE the near and the far value,
// bit for bit.  An unused slot holds the inverted box (3e38, -3e38) (host/bvh_wide.hpp): near > far on every axis, so it fails
// tn <= tf without a look at its reference.
// node + byte offset (0 / 16), added to the node's address once it is formed (left to nvcc, the sum is re-associated into three wide
// multiplies and six 64-bit adds per visit; this form costs two instructions per address and three registers per ray)
RT_DEV const float4* wide_row(const float4* node, uint32_t byte_off) {
#ifdef __CUDA_ARCH__
    unsigned long long a;
    asm("mad.wide.u32 %0, %1, 1, %2;" : "=l"(a) : "r"(byte_off), "l"(reinterpret_cast<unsigned long long>(node)));
    return reinterpret_cast<const float4*>(a);
#else
    return reinterpret_cast<const float4*>(reinterpret_cast<const char*>(node) + byte_off);
#endif
}
RT_DEV unsigned long long wide_key_nf(float nx, float fx, float ny, float fy, float nz, float fz, float ref, const RayF& f, float t_min, float t_max) {
    const float xn = fmaf(nx, f.idx, -f.oodx), xf = fmaf(fx, f.idx, -f.oodx);
    const float yn = fmaf(ny, f.idy, -f.oody), yf = fmaf(fy, f.idy, -f.oody);
    const float zn = fmaf(nz, f.idz, -f.oodz), zf = fmaf(fz, f.idz, -f.oodz);
    const float tn = fmaxf(fmaxf(xn, yn), fmaxf(zn, t_min));
    const float tf = fminf(fminf(xf, yf), fminf(zf, t_max));
    if (!(tn <= tf)) return ~0ull;
    return ((unsigned long long)(__float_as_uint(tn) & 0x7fffffffu) << 32) | (unsigned long long)__float_as_uint(ref);
}
RT_DEV float4 wide_lerp(float4 v, float4 d, float ms) { return make_float4(fmaf(d.x, ms, v.x), fmaf(d.y, ms, v.y), fmaf(d.z, ms, v.z), fmaf(d.w, ms, v.w)); }
// The near and far row of one axis (q = the node's row pair of that axis, sg = the ray's byte offset of its near row); `motion`: the
// rows of the motion nodes (DeviceScene::mnodes4) interpolated to the ray's shutter position ms
RT_DEV void wide_rows(const float4* q, uint32_t sg, bool motion, float ms, float4& n, float4& fr) {
    const float4* qn = wide_row(q, sg);
    const float4* qf = wide_row(q, sg ^ 16u);
    n = __ldg(qn); fr = __ldg(qf);
    if (motion) { n = wide_lerp(n, __ldg(qn + 8), ms); fr = wide_lerp(fr, __ldg(qf + 8), ms); }
}
// The signed-row key of the four children of a node, an axis at a time: fmaxf / fminf return one of their operands (the non-NaN one),
// so the running max(max(max(x, t_min), y), z) is the value of max(max(x, y), max(z, t_min)) (up to the sign of a zero, which the key
// masks off and tn <= tf does not see): the same keys, bit for bit
RT_DEV void wide_fold_x(const float4& n, const float4& fr, const RayF& f, float t_min, float t_max, float4& tn, float4& tf) {
    tn.x = fmaxf(fmaf(n.x, f.idx, -f.oodx), t_min); tf.x = fminf(fmaf(fr.x, f.idx, -f.oodx), t_max);
    tn.y = fmaxf(fmaf(n.y, f.idx, -f.oodx), t_min); tf.y = fminf(fmaf(fr.y, f.idx, -f.oodx), t_max);
    tn.z = fmaxf(fmaf(n.z, f.idx, -f.oodx), t_min); tf.z = fminf(fmaf(fr.z, f.idx, -f.oodx), t_max);
    tn.w = fmaxf(fmaf(n.w, f.idx, -f.oodx), t_min); tf.w = fminf(fmaf(fr.w, f.idx, -f.oodx), t_max);
}
RT_DEV void wide_fold(const float4& n, const float4& fr, float id, float ood, float4& tn, float4& tf) {
    tn.x = fmaxf(tn.x, fmaf(n.x, id, -ood)); tf.x = fminf(tf.x, fmaf(fr.x, id, -ood));
    tn.y = fmaxf(tn.y, fmaf(n.y, id, -ood)); tf.y = fminf(tf.y, fmaf(fr.y, id, -ood));
    tn.z = fmaxf(tn.z, fmaf(n.z, id, -ood)); tf.z = fminf(tf.z, fmaf(fr.z, id, -ood));
    tn.w = fmaxf(tn.w, fmaf(n.w, id, -ood)); tf.w = fminf(tf.w, fmaf(fr.w, id, -ood));
}
RT_DEV unsigned long long wide_key_tn(float tn, float tf, float ref) {
    if (!(tn <= tf)) return ~0ull;
    return ((unsigned long long)(__float_as_uint(tn) & 0x7fffffffu) << 32) | (unsigned long long)__float_as_uint(ref);
}
#ifndef RT_WIDE_CE32
#define RT_WIDE_CE32 1
#endif
#define RT_WIDE_MISS(k) (RT_WIDE_CE32 ? (uint32_t)((k) >> 32) == 0xffffffffu : (k) == ~0ull) // a hit's distance bits are never all ones
RT_DEV void wide_ce(unsigned long long& a, unsigned long long& b) {
    // ordered by the distance word alone: equal distances may come out either way, which only the visiting order sees
    const bool s = RT_WIDE_CE32 ? (uint32_t)(a >> 32) > (uint32_t)(b >> 32) : a > b;
    const unsigned long long lo = s ? b : a, hi = s ? a : b;
    a = lo; b = hi;
}
// The walk's stack is reached through wstk_put / wstk_get so that it can be something else than a plain local-memory array: the host
// emulation counts the accesses per depth with it (tests/host_emul: book-1 never goes past 8 entries, the 871 200-triangle mesh past 19),
// and round 2 measured a variant with the first 8 / 12 / 16 entries per thread in shared memory ([entry][thread], conflict free):
// book-1 final -3.6 %, mesh -1 ... +1.3 % (profiles/r2_50_ab_signed_rows_smem_stack.txt) - the local-memory stack is not what the
// pop stalls on, so it stays.
RT_DEV void wstk_put(unsigned long long* s, int i, unsigned long long v) { s[i] = v; }
RT_DEV unsigned long long wstk_get(const unsigned long long* s, int i) { return s[i]; }
template <class STK> RT_DEV uint32_t wide_pop(const STK& stack, int& sp, float tmaxf) {
    while (sp) {
        const unsigned long long e = wstk_get(stack, --sp);
        if ((uint32_t)(e >> 32) <= __float_as_uint(tmaxf)) return (uint32_t)e; // both non-negative floats: integer compare
    }
    return 0xffffffffu;
}
// RESUME = true: the resumable form used by k_mega_r (see trace_resume below): state (cur, sp, stack, best) lives in the
// caller, called by all 32 lanes, returns once `wait_thresh` of the lanes that entered with work have finished.
// RESUME = false: walks until this lane is done.
// walk_wide: the per-ray constants come from the caller (see walk_pairs); trace_wide below derives them per call.
template <uint32_t PM, bool RESUME, bool COUNT = false, class STK>
RT_DEV void walk_wide(const DeviceScene& S, const Ray& r, const RayF& f, const RayPre& pre, double t_min, BestHit& best, uint32_t& cur, int& sp, STK& stack,
                      uint32_t wait_thresh, uint32_t inst = 0u, TraceCounters* cnt = nullptr) {
    const unsigned full = 0xffffffffu;
    const float tminf = fmaxf(f32_down(t_min), 0.f);
    float tmaxf = f32_up(best.t);
    const float4* __restrict__ nodes4 = S.nodes4;
    // spheres + moving spheres: motion-interpolated child boxes (DeviceScene::mnodes4), as trace_instance does with mnodes
    const float4* __restrict__ mnodes4 = S.mnodes4;
    const bool MOTION = PM == 0x3u && mnodes4 != nullptr;
    float ms = 0.f;
    if (MOTION) { const double sd = (r.time - S.motion_t0) * S.motion_inv_dt; ms = (float)(sd < 0.0 ? 0.0 : (sd > 1.0 ? 1.0 : sd)); }
    // byte offset of the row the ray enters through, per axis (0 = lo, 16 = hi)
    uint32_t sgx = f.idx < 0.f ? 16u : 0u, sgy = f.idy < 0.f ? 16u : 0u, sgz = f.idz < 0.f ? 16u : 0u;
    const uint32_t DONE = 0xffffffffu;
    uint32_t n0 = 0;
    if (RESUME) n0 = __popc(__ballot_sync(full, cur != DONE));
    for (;;) {
        // Bounded node loop: a lane takes at most INNER node steps before the warp looks at the leaves that are pending.  Unbounded
        // (the classic while-while) every lane that already holds a leaf idles until the slowest lane of the warp has found one; one
        // step at a time (if-if) the leaf code is issued every iteration for few lanes.  Measured, same box (profiles/r2_41_ab_inner.txt):
        // sphere scenes are best at 1 (book-1 final 86.9 -> 83.5 ms), the 871 200-triangle mesh at 6 (58.3 -> 52.0 ms per 10 spp).
#ifndef RT_INNER_SPH
#define RT_INNER_SPH 1
#endif
#ifndef RT_INNER_TRI
#define RT_INNER_TRI 6
#endif
#ifndef RT_INNER_MEDIA
#define RT_INNER_MEDIA 1 // the media wavefront kernels' masks (rects + boxes, + spheres + moving spheres): 1 / 2 / unbounded measured, 1 is best
#endif
        constexpr int INNER = RT_PM_HAS(PM, PRIM_TRI) ? RT_INNER_TRI : ((PM == 0x18u || PM == 0x1bu) ? RT_INNER_MEDIA : RT_INNER_SPH);
        // The sphere kernels (k_mega at 80 registers) load and fold the node one axis at a time: fewer rows live at once.  The triangle
        // and media kernels keep all seven rows in flight (the fold measured -2.9 % on the 871 200-triangle mesh, -0.7 % on book-2 final)
        constexpr bool WIDE_FOLD = PM == 0x1u || PM == 0x3u || PM == 0x5u;
#pragma unroll 1
        for (int inner = 0; inner < INNER && cur != DONE && !(cur & RT_LEAF_FLAG); ++inner) {
            unsigned long long k0, k1, k2, k3;
            if constexpr (RT_WIDE_SIGNED && WIDE_FOLD) { // rows picked by the ray's direction signs: near = the planes it enters through, far = leaves through
                if (COUNT) cnt->nodes += 4;
                // MOTION: box(t) = box at the shutter's start + s * delta, 256 bytes per node (start and end boxes are valid and the
                // interpolation is monotonic, so lo(t) <= hi(t) holds and the signed rows stay right)
                const float4* __restrict__ q = MOTION ? mnodes4 + 16 * (size_t)cur : nodes4 + 8 * (size_t)cur;
                // one axis at a time, folded into running near / far values: a pair of rows is dead before the next one is needed
                float4 n, fr, tn, tf;
                wide_rows(q, sgx, MOTION, ms, n, fr);
                wide_fold_x(n, fr, f, tminf, tmaxf, tn, tf);
                wide_rows(q + 2, sgy, MOTION, ms, n, fr);
                wide_fold(n, fr, f.idy, f.oody, tn, tf);
                wide_rows(q + 4, sgz, MOTION, ms, n, fr);
                wide_fold(n, fr, f.idz, f.oodz, tn, tf);
                const float4 rf = __ldg(q + 6);
                k0 = wide_key_tn(tn.x, tf.x, rf.x);
                k1 = wide_key_tn(tn.y, tf.y, rf.y);
                k2 = wide_key_tn(tn.z, tf.z, rf.z);
                k3 = wide_key_tn(tn.w, tf.w, rf.w);
            } else {
                float4 lx, hx, ly, hy, lz, hz, rf;
                if (MOTION) { // box(t) = box at the shutter's start + s * delta: 256 bytes per node
                    // (signed rows as below: start and end boxes are valid and the interpolation is monotonic, so lo(t) <= hi(t) holds)
                    const float4* __restrict__ q = mnodes4 + 16 * (size_t)cur;
                    const float4* qx = RT_WIDE_SIGNED ? wide_row(q, sgx) : q;
                    const float4* qX = RT_WIDE_SIGNED ? wide_row(q, sgx ^ 16u) : q + 1;
                    const float4* qy = RT_WIDE_SIGNED ? wide_row(q, sgy) + 2 : q + 2;
                    const float4* qY = RT_WIDE_SIGNED ? wide_row(q, sgy ^ 16u) + 2 : q + 3;
                    const float4* qz = RT_WIDE_SIGNED ? wide_row(q, sgz) + 4 : q + 4;
                    const float4* qZ = RT_WIDE_SIGNED ? wide_row(q, sgz ^ 16u) + 4 : q + 5;
                    lx = __ldg(qx); hx = __ldg(qX); ly = __ldg(qy); hy = __ldg(qY); lz = __ldg(qz); hz = __ldg(qZ); rf = __ldg(q + 6);
                    const float4 dlx = __ldg(qx + 8), dhx = __ldg(qX + 8), dly = __ldg(qy + 8), dhy = __ldg(qY + 8), dlz = __ldg(qz + 8), dhz = __ldg(qZ + 8);
                    lx.x = fmaf(dlx.x, ms, lx.x); lx.y = fmaf(dlx.y, ms, lx.y); lx.z = fmaf(dlx.z, ms, lx.z); lx.w = fmaf(dlx.w, ms, lx.w);
                    hx.x = fmaf(dhx.x, ms, hx.x); hx.y = fmaf(dhx.y, ms, hx.y); hx.z = fmaf(dhx.z, ms, hx.z); hx.w = fmaf(dhx.w, ms, hx.w);
                    ly.x = fmaf(dly.x, ms, ly.x); ly.y = fmaf(dly.y, ms, ly.y); ly.z = fmaf(dly.z, ms, ly.z); ly.w = fmaf(dly.w, ms, ly.w);
                    hy.x = fmaf(dhy.x, ms, hy.x); hy.y = fmaf(dhy.y, ms, hy.y); hy.z = fmaf(dhy.z, ms, hy.z); hy.w = fmaf(dhy.w, ms, hy.w);
                    lz.x = fmaf(dlz.x, ms, lz.x); lz.y = fmaf(dlz.y, ms, lz.y); lz.z = fmaf(dlz.z, ms, lz.z); lz.w = fmaf(dlz.w, ms, lz.w);
                    hz.x = fmaf(dhz.x, ms, hz.x); hz.y = fmaf(dhz.y, ms, hz.y); hz.z = fmaf(dhz.z, ms, hz.z); hz.w = fmaf(dhz.w, ms, hz.w);
                } else if (RT_WIDE_SIGNED) { // rows picked by the ray's direction signs: l* = the planes it enters through, h* = leaves through
                    const float4* __restrict__ q = nodes4 + 8 * (size_t)cur;
                    lx = __ldg(wide_row(q, sgx)); hx = __ldg(wide_row(q, sgx ^ 16u)); ly = __ldg(wide_row(q, sgy) + 2); hy = __ldg(wide_row(q, sgy ^ 16u) + 2);
                    lz = __ldg(wide_row(q, sgz) + 4); hz = __ldg(wide_row(q, sgz ^ 16u) + 4); rf = __ldg(q + 6);
                } else {
                    const float4* __restrict__ q = nodes4 + 8 * (size_t)cur;
                    lx = __ldg(q); hx = __ldg(q + 1); ly = __ldg(q + 2); hy = __ldg(q + 3); lz = __ldg(q + 4); hz = __ldg(q + 5); rf = __ldg(q + 6);
                }
                if (COUNT) cnt->nodes += 4;
                if (RT_WIDE_SIGNED) {
                    k0 = wide_key_nf(lx.x, hx.x, ly.x, hy.x, lz.x, hz.x, rf.x, f, tminf, tmaxf);
                    k1 = wide_key_nf(lx.y, hx.y, ly.y, hy.y, lz.y, hz.y, rf.y, f, tminf, tmaxf);
                    k2 = wide_key_nf(lx.z, hx.z, ly.z, hy.z, lz.z, hz.z, rf.z, f, tminf, tmaxf);
                    k3 = wide_key_nf(lx.w, hx.w, ly.w, hy.w, lz.w, hz.w, rf.w, f, tminf, tmaxf);
                } else {
                    k0 = wide_key(lx.x, hx.x, ly.x, hy.x, lz.x, hz.x, rf.x, f, tminf, tmaxf);
                    k1 = wide_key(lx.y, hx.y, ly.y, hy.y, lz.y, hz.y, rf.y, f, tminf, tmaxf);
                    k2 = wide_key(lx.z, hx.z, ly.z, hy.z, lz.z, hz.z, rf.z, f, tminf, tmaxf);
                    k3 = wide_key(lx.w, hx.w, ly.w, hy.w, lz.w, hz.w, rf.w, f, tminf, tmaxf);
                }
            }
            // Only the nearest child is found exactly (three compare-exchanges); k1..k3 are pushed as they are.  The full five-exchange
            // sort (far-to-near pushes) measured 2.7 % slower on book-1 final and 3 % on the 871 200-triangle mesh (profiles/r2_00_ab.log):
            // an entry that a nearer hit has culled is dropped when popped, so the order of the queued ones matters little.
            wide_ce(k0, k1); wide_ce(k2, k3); wide_ce(k0, k2);
            if (!RT_WIDE_MISS(k3)) wstk_put(stack, sp++, k3);
            if (!RT_WIDE_MISS(k2)) wstk_put(stack, sp++, k2);
            if (!RT_WIDE_MISS(k1)) wstk_put(stack, sp++, k1);
            cur = !RT_WIDE_MISS(k0) ? (uint32_t)k0 : wide_pop(stack, sp, tmaxf);
        }
        if (cur != DONE && (cur & RT_LEAF_FLAG)) { // a leaf reference
            if (COUNT) cnt->prims += ((cur >> 25) & 7u) + 1u;
            leaf_test<PM>(S, r, pre, t_min, best, (cur >> 28) & 7u, cur & 0x1ffffffu, ((cur >> 25) & 7u) + 1u, inst);
            tmaxf = f32_up(best.t);
            cur = wide_pop(stack, sp, tmaxf);
        }
        if (RESUME) {
            const uint32_t still = __popc(__ballot_sync(full, cur != DONE));
            if (still == 0 || n0 - still >= wait_thresh) break;
        } else if (cur == DONE) {
            break;
        }
    }
}

template <uint32_t PM, bool RESUME, bool COUNT = false, class STK>
RT_DEV void trace_wide(const DeviceScene& S, const Ray& r, double t_min, BestHit& best, uint32_t& cur, int& sp, STK& stack, uint32_t wait_thresh,
                       uint32_t inst = 0u, TraceCounters* cnt = nullptr) {
    const RayF f = make_rayf(r);
    const RayPre pre = make_raypre(r, (PM & 0x18u) != 0 && (S.flags & 1u) != 0);
    walk_wide<PM, RESUME, COUNT>(S, r, f, pre, t_min, best, cur, sp, stack, wait_thresh, inst, cnt);
}

RT_DEV bool inst_box_hit(const Instance* ip, const Ray& r, double t_min, double t_max) {
    const RayF f = make_rayf(r);
    float tn;
    const float4 lo = make_float4(__ldg(&ip->bmin[0]), __ldg(&ip->bmin[1]), __ldg(&ip->bmin[2]), 0.f);
    const float4 hi = make_float4(__ldg(&ip->bmax[0]), __ldg(&ip->bmax[1]), __ldg(&ip->bmax[2]), 0.f);
    return slab(lo, hi, f, f32_down(t_min), f32_up(t_max), tn);
}

// world.hit restricted to the instances [i0, i1): the main world or one medium's boundary.
// XF = false: the scene has no Translate / RotateY wrappers (every chain is empty): no ray transform going in,
// no chain unwinding coming out
// WIDE = true (main world only, t_min >= 0; the host built Instance::root4 for every instance of the range): the 4-wide walk
template <bool COUNT, uint32_t PM = RT_PM_ALL, bool XF = true, bool WIDE = false>
RT_DEV void trace_instances(const DeviceScene& S, uint32_t i0, uint32_t i1, const Ray& world_ray, double t_min, BestHit& best, TraceCounters* cnt) {
    for (uint32_t i = i0; i < i1; ++i) {
        const Instance* ip = &S.instances[i];
        Ray r = world_ray;
        if (XF) xform_ray(S.ops, __ldg(&ip->chain_off), __ldg(&ip->chain_len), r);
        if (WIDE) {
            unsigned long long wstack[RT_WIDE_STACK];
            uint32_t cur = __ldg(&ip->root4);
            int sp = 0;
            trace_wide<PM, false, COUNT>(S, r, t_min, best, cur, sp, wstack, 0u, i, cnt);
        } else if (PM == 0x18u) trace_instance_spec<COUNT, PM>(S, i, r, t_min, best, cnt);
        else trace_instance<COUNT, PM>(S, i, r, t_min, best, cnt);
    }
}

// ------------------------------------------------------------------ hit record (hit.rs:9-18)
struct HitRec {
    D3 p, n;
    double t, u, v;
    uint32_t mat, prim_id;
    bool front;
};
RT_DEV void face_forward(D3 dir, D3 outward, D3& n, bool& front) { // hit.rs:69-79
    front = dot(dir, outward) < 0.0;
    n = front ? outward : -outward;
}
RT_DEV void sphere_uv(D3 p, double& u, double& v) { // hit.rs:195-200
    const double PI = 3.14159265358979323846264338327950288;
    const double theta = acos(-p.y);
    const double phi = atan2(-p.z, p.x) + PI;
    u = phi / (2.0 * PI);
    v = theta / PI;
}

// Rebuild the full HitRecord of the winning primitive, then undo the wrapper chain from the inside
// out exactly as Translate::hit / RotateY::hit do (hit.rs:808-820, 909-930), including their
// re-face-forwarding quirks (SURVEY.md Appendix A8).
// UVMODE: 0 = never compute sphere (u,v) (the scene has no image texture), 1 = always (parity hook),
// 2 = when the hit material's texture chain reads them
template <int UVMODE, uint32_t PM = RT_PM_ALL, bool XF = true>
RT_DEV HitRec finalize_hit(const DeviceScene& S, const Ray& world_ray, const BestHit& b) {
    HitRec h;
    const Instance* ip = &S.instances[b.inst];
    uint32_t coff = 0, clen = 0;
    if (XF) { coff = __ldg(&ip->chain_off); clen = __ldg(&ip->chain_len); }
    Ray r = world_ray;
    if (XF) xform_ray(S.ops, coff, clen, r);
    const PrimMeta m = S.meta[b.type][b.idx];
    h.mat = m.mat_id;
    h.prim_id = m.prim_id + b.side;
    h.t = b.t;
    h.p = ray_at(r, b.t);
    h.u = 0.0; h.v = 0.0;
    D3 outward = mk3(0, 1, 0);
    const uint32_t ty = b.type;
    if (RT_PM_HAS(PM, PRIM_SPHERE) && ((PM & ~1u) == 0 || ty == PRIM_SPHERE)) {
        const DSphere s = S.spheres[b.idx];
        outward = (h.p - mk3(s.cx, s.cy, s.cz)) * (1.0 / s.r);
        if (UVMODE != 0) {
            bool need_uv = UVMODE == 1;
            if (UVMODE == 2) need_uv = (__ldg(&S.materials[m.mat_id].flags) & 1u) != 0;
            if (need_uv) sphere_uv(outward, h.u, h.v);
        }
    } else if (RT_PM_HAS(PM, PRIM_MOVING) && ty == PRIM_MOVING) {
        const DMoving s = S.movings[b.idx];
        outward = (h.p - moving_center(s, r.time)) * (1.0 / s.r); // u = v = 0 (hit.rs:310-311)
    } else if (RT_PM_HAS(PM, PRIM_GRAVITY) && ty == PRIM_GRAVITY) {
        const DGravity s = S.gravities[b.idx];
        outward = (h.p - gravity_center(S, s, r.time)) * (1.0 / s.r);
    } else if (RT_PM_HAS(PM, PRIM_RECT) && ty == PRIM_RECT) {
        const DRect q = S.rects[b.idx];
        const int ax = q.axis, ia = ax == 0 ? 1 : 0, ib = ax == 2 ? 1 : 2;
        h.u = (axis_of(h.p, ia) - q.a0) / (q.a1 - q.a0); // hit.rs:486-487 (x, y recomputed as o + t*d = p)
        h.v = (axis_of(h.p, ib) - q.b0) / (q.b1 - q.b0);
        outward = mk3(ax == 0 ? 1.0 : 0.0, ax == 1 ? 1.0 : 0.0, ax == 2 ? 1.0 : 0.0);
    } else if (RT_PM_HAS(PM, PRIM_BOX) && ty == PRIM_BOX) {
        const DBox q = S.boxes[b.idx];
        const int s = (int)b.side;
        const int ax = s < 2 ? 2 : (s < 4 ? 1 : 0), ia = ax == 0 ? 1 : 0, ib = ax == 2 ? 1 : 2;
        h.u = (axis_of(h.p, ia) - q.p0[ia]) / (q.p1[ia] - q.p0[ia]);
        h.v = (axis_of(h.p, ib) - q.p0[ib]) / (q.p1[ib] - q.p0[ib]);
        outward = mk3(ax == 0 ? 1.0 : 0.0, ax == 1 ? 1.0 : 0.0, ax == 2 ? 1.0 : 0.0);
    } else if (RT_PM_HAS(PM, PRIM_TRI)) { // PRIM_TRI: u = v = 1 (hit.rs:157-158)
        const DTri* tp = &S.tris[b.idx];
        const float4 q2 = __ldg(reinterpret_cast<const float4*>(tp) + 2);
        outward = mk3(q2.y, q2.z, q2.w);
        h.u = 1.0; h.v = 1.0;
    }
    face_forward(r.d, outward, h.n, h.front);
    // unwind the chain: r currently holds the innermost ray
    D3 d_in = r.d;
    for (int i = XF ? (int)clen - 1 : -1; i >= 0; --i) {
        const XformOp op = S.ops[coff + i];
        if (op.type == XF_TRANSLATE) {
            h.p = mk3(h.p.x + op.a, h.p.y + op.b, h.p.z + op.c);
            face_forward(d_in, h.n, h.n, h.front); // against moved_r (same direction), hit.rs:810
        } else {
            const double s = op.a, c = op.b;
            h.p = mk3(c * h.p.x + s * h.p.z, h.p.y, -s * h.p.x + c * h.p.z);
            const D3 nw = mk3(c * h.n.x + s * h.n.z, h.n.y, -s * h.n.x + c * h.n.z);
            face_forward(d_in, nw, h.n, h.front); // world normal against the OBJECT-space ray, hit.rs:921
            d_in = mk3(c * d_in.x + s * d_in.z, d_in.y, -s * d_in.x + c * d_in.z); // direction one level out
        }
    }
    return h;
}

// ------------------------------------------------------------------ ConstantMedium::hit (hit.rs:955-986)
// GENERAL = false compiles out the two-traversal path for arbitrary boundaries (it costs the hot
// kernels registers and a second traversal stack); the host only picks such kernels when every medium
// of the scene has the single-sphere / single-box fast path (DeviceScene.flags bit 1).
template <bool COUNT, bool GENERAL>
RT_DEV void medium_query(const DeviceScene& S, uint32_t mi, const Ray& world_ray, double t_min, double& closest, int32_t& winner, D3& p_out,
                         uint64_t seed, uint64_t path_id, uint32_t segment, TraceCounters* cnt) {
    const Medium md = S.media[mi];
    Ray r = world_ray;
    xform_ray(S.ops, md.chain_off, md.chain_len, r);
    // boundary.hit(r, -inf, +inf) then boundary.hit(r, rec1.t + 0.0001, +inf) (hit.rs:956-957)
    double ta, tb;
    if (md.fast_type != 0) {
        // the boundary is a single sphere or a single box (optionally under Translate/RotateY): both
        // crossings from one solve instead of two traversals
        Ray rb = r;
        xform_ray(S.ops, md.fast_chain_off, md.fast_chain_len, rb);
        if (COUNT) cnt->prims += 2;
        if (md.fast_type == 1) {
            const DSphere sp = S.spheres[md.fast_idx];
            const D3 oc = rb.o - mk3(sp.cx, sp.cy, sp.cz);
            const double a = length_squared(rb.d), half_b = dot(oc, rb.d);
            const double disc = fma(half_b, half_b, -(a * fma(-sp.r, sp.r, length_squared(oc))));
            if (disc < 0.0) return;
            const double sq = sqrt(disc), inv_a = 1.0 / a;
            ta = (-half_b - sq) * inv_a;
            tb = (-half_b + sq) * inv_a;
            if (!(ta < RT_INF) || !(ta > -RT_INF)) return;
            if (tb < ta + 0.0001 || !(tb < RT_INF)) return;
        } else {
            const DBox bx = S.boxes[md.fast_idx];
            const RayPre pre = make_raypre(rb, true);
            double ts[6];
            ta = RT_INF;
#pragma unroll
            for (int sd = 0; sd < 6; ++sd) { ts[sd] = box_side_t(rb, pre, bx, sd); ta = fmin(ta, ts[sd]); }
            if (!(ta < RT_INF)) return;
            tb = RT_INF;
#pragma unroll
            for (int sd = 0; sd < 6; ++sd) if (ts[sd] >= ta + 0.0001) tb = fmin(tb, ts[sd]);
            if (!(tb < RT_INF)) return;
        }
    } else if (GENERAL) {
        BestHit b1;
        best_init(b1, RT_INF);
        trace_instances<COUNT>(S, md.inst_begin, md.inst_end, r, -RT_INF, b1, cnt);
        if (b1.type == RT_NONE) return;
        BestHit b2;
        best_init(b2, RT_INF);
        trace_instances<COUNT>(S, md.inst_begin, md.inst_end, r, b1.t + 0.0001, b2, cnt);
        if (b2.type == RT_NONE) return;
        ta = b1.t; tb = b2.t;
    } else {
        return; // kernels compiled without the general path are only launched when every medium has the fast path
    }
    double t1 = fmax(ta, t_min);
    const double t2 = fmin(tb, closest);
    if (t1 >= t2) return;
    if (t1 < 0.0) t1 = 0.0;
    const double ray_length = sqrt(length_squared(r.d));
    const double distance_inside_boundary = (t2 - t1) * ray_length;
    const double hit_distance = md.neg_inv_density * log(medium_xi(seed, path_id, md.prim_id, segment));
    if (hit_distance > distance_inside_boundary) return;
    const double t = t1 + hit_distance / ray_length;
    if (!(t <= closest)) return;
    closest = t;
    winner = (int32_t)mi;
    // p = r.at(t) in the medium's space, brought back out through the medium's own chain
    D3 p = ray_at(r, t);
    for (int i = (int)md.chain_len - 1; i >= 0; --i) {
        const XformOp op = S.ops[md.chain_off + i];
        if (op.type == XF_TRANSLATE) p = mk3(p.x + op.a, p.y + op.b, p.z + op.c);
        else p = mk3(op.b * p.x + op.a * p.z, p.y, -op.a * p.x + op.b * p.z);
    }
    p_out = p;
}

// rec.p of a medium hit at parameter t (hit.rs:976): r.at(t) in the medium's own space, brought out through the medium's chain -
// the same operations, in the same order, as the tail of medium_query (k_pool rebuilds the record when it shades the slot)
RT_DEV D3 medium_point(const DeviceScene& S, const Medium& md, const Ray& world_ray, double t) {
    Ray r = world_ray;
    xform_ray(S.ops, md.chain_off, md.chain_len, r);
    D3 p = ray_at(r, t);
    for (int i = (int)md.chain_len - 1; i >= 0; --i) {
        const XformOp op = S.ops[md.chain_off + i];
        if (op.type == XF_TRANSLATE) p = mk3(p.x + op.a, p.y + op.b, p.z + op.c);
        else p = mk3(op.b * p.x + op.a * p.z, p.y, -op.a * p.x + op.b * p.z);
    }
    return p;
}

// world.hit(ray, t_min, t_max) (world.rs:68): surfaces first, then every medium against the closest
// surface (order independent because medium draws are keyed, SURVEY.md Appendix D5).
template <bool COUNT, int UVMODE, bool MEDIA, bool GENERAL_MEDIA = true, uint32_t PM = RT_PM_ALL, bool XF = true, bool WIDE = false>
RT_DEV bool world_hit(const DeviceScene& S, const Ray& ray, double t_min, double t_max, bool media, uint64_t seed, uint64_t path_id, uint32_t segment,
                      HitRec& h, TraceCounters* cnt) {
    BestHit best;
    best_init(best, t_max);
    trace_instances<COUNT, PM, XF, WIDE>(S, 0, S.n_main_instances, ray, t_min, best, cnt);
    if (MEDIA) {
        double closest = best.t;
        int32_t mwin = -1;
        D3 mp = mk3(0, 0, 0);
        if (media) {
            for (uint32_t mi = 0; mi < S.n_media; ++mi) medium_query<COUNT, GENERAL_MEDIA>(S, mi, ray, t_min, closest, mwin, mp, seed, path_id, segment, cnt);
        }
        if (mwin >= 0) {
            const Medium md = S.media[mwin];
            h.p = mp; h.n = mk3(0, 0, 0); h.t = closest; h.u = 0.0; h.v = 0.0; h.front = true; // hit.rs:975-984
            h.mat = md.mat_id; h.prim_id = md.prim_id;
            return true;
        }
    }
    if (best.type == RT_NONE) return false;
    h = finalize_hit<UVMODE, PM, XF>(S, ray, best);
    return true;
}

// ------------------------------------------------------------------ perlin.rs / texture.rs
struct F3 { float x, y, z; };
RT_DEV F3 mkf3(float x, float y, float z) { F3 r; r.x = x; r.y = y; r.z = z; return r; }

RT_DEV double perlin_noise(const PerlinTable* __restrict__ pt, D3 p) { // perlin.rs:28-52, 85-106
    const double fx = floor(p.x), fy = floor(p.y), fz = floor(p.z);
    const double u = p.x - fx, v = p.y - fy, w = p.z - fz;
    const int i = (int)fx, j = (int)fy, k = (int)fz;
    const double uu = u * u * (3.0 - 2.0 * u), vv = v * v * (3.0 - 2.0 * v), ww = w * w * (3.0 - 2.0 * w);
    double accum = 0.0;
#pragma unroll
    for (int di = 0; di < 2; ++di)
#pragma unroll
        for (int dj = 0; dj < 2; ++dj)
#pragma unroll
            for (int dk = 0; dk < 2; ++dk) {
                const int idx = pt->perm_x[(i + di) & 255] ^ pt->perm_y[(j + dj) & 255] ^ pt->perm_z[(k + dk) & 255];
                const double cx = pt->ranvec[idx][0], cy = pt->ranvec[idx][1], cz = pt->ranvec[idx][2];
                const double wx = u - di, wy = v - dj, wz = w - dk;
                accum += (di ? uu : (1.0 - uu)) * (dj ? vv : (1.0 - vv)) * (dk ? ww : (1.0 - ww)) * (cx * wx + cy * wy + cz * wz);
            }
    return accum;
}
RT_DEV double perlin_turbulence(const PerlinTable* __restrict__ pt, D3 p, int depth) { // perlin.rs:54-66
    double accum = 0.0, weight = 1.0;
    D3 tp = p;
    for (int o = 0; o < depth; ++o) {
        accum += weight * perlin_noise(pt, tp);
        weight *= 0.5;
        tp = tp * 2.0;
    }
    return fabs(accum);
}

// FULL = false compiles only SolidColor and Checker (kernels picked for scenes without Noise / Image
// textures: the Perlin and image code would only cost instruction-cache space)
// perlin0 = the scene's first Perlin table staged in shared memory by the caller (k_shade_all), or nullptr
template <bool FULL = true>
RT_DEV F3 tex_value(const DeviceScene& S, uint32_t tex, double u, double v, D3 p, const PerlinTable* perlin0 = nullptr) { // texture.rs:7-9
    for (int guard = 0; guard < 64; ++guard) {
        const DTexture* t = &S.textures[tex];
        const uint32_t type = __ldg(&t->type);
        if (type == TEX_SOLID) return mkf3(__ldg(&t->rgb[0]), __ldg(&t->rgb[1]), __ldg(&t->rgb[2])); // texture.rs:27-31
        if (type == TEX_CHECKER) { // texture.rs:54-64: sign of sin(10x) sin(10y) sin(10z)
            const double sines = sin(10.0 * p.x) * sin(10.0 * p.y) * sin(10.0 * p.z); // f64 like the reference: an f32 argument moves the checker boundaries by ~5e-4 rad at |10 p| ~ 1e4
            tex = sines < 0.0 ? __ldg(&t->b) : __ldg(&t->a);
            continue;
        }
        if (!FULL) break;
        if (type == TEX_NOISE) { // texture.rs:80-88
            const uint32_t pi = __ldg(&t->a);
            const PerlinTable* pt = (perlin0 && pi == 0u) ? perlin0 : &S.perlin[pi];
            const double s = 0.5 * (1.0 + sin(t->scale * p.z + 10.0 * perlin_turbulence(pt, p, 7)));
            return mkf3((float)s, (float)s, (float)s);
        }
        // TEX_IMAGE, texture.rs:102-121: nearest texel, row 0 = top of file, v flipped
        double uc = u < 0.0 ? 0.0 : (u > 1.0 ? 1.0 : u);
        double vc = v < 0.0 ? 0.0 : (v > 1.0 ? 1.0 : v);
        vc = 1.0 - vc;
        const int W = (int)t->w, H = (int)t->h;
        int i = (int)(uc * (double)W), j = (int)(vc * (double)H);
        i = min(i, W - 1); j = min(j, H - 1);
        const float4 px = __ldg(&S.texels[t->a + (size_t)j * W + i]);
        const float cs = 1.0f / 255.0f;
        return mkf3(cs * px.x, cs * px.y, cs * px.z);
    }
    return mkf3(0.f, 0.f, 0.f);
}

// world.rs:86-89: what a miss contributes per unit of throughput.  Constant `background`, or the book-1 sky of the revision that
// rendered images/book1.png (rt_scene_set_background_gradient): (1 - t) * horizon + t * zenith, t = 0.5 * (unit(d).y + 1).
RT_DEV F3 miss_color(const DeviceScene& S, D3 d) {
    if (!S.bg_gradient) return mkf3(S.background[0], S.background[1], S.background[2]);
    const float t = (float)(0.5 * (unit(d).y + 1.0)), w = 1.0f - t;
    return mkf3(w * S.background[0] + t * S.background_top[0], w * S.background[1] + t * S.background_top[1], w * S.background[2] + t * S.background_top[2]);
}

// ------------------------------------------------------------------ Material::scatter (hit.rs:1004-1152)
// Returns true when the path continues; `dir` = scattered direction, `att` = attenuation.
// Lambertian, Metal and Isotropic all start with random_in_unit_sphere (hit.rs:1033, 1068, 1007); the *_finish halves take its
// result `rs`, so that the fused kernels can run ONE rejection loop for every lane of a warp that needs one, whatever its material
// (book-1: a second, metal-only loop of 4-5 diverged iterations per warp and segment otherwise)
template <bool FULLTEX = true>
RT_DEV bool lambertian_finish(const DeviceScene& S, const DMaterial& m, D3 p, D3 n, double u, double v, D3 rs, D3& dir, F3& att,
                              const PerlinTable* perlin0 = nullptr) {
    D3 sd = n + unit(rs); // random_unit_vector, vec3.rs:297-299
    if (near_zero(sd)) sd = n;
    dir = sd;
    att = tex_value<FULLTEX>(S, m.tex, u, v, p, perlin0);
    return true;
}
RT_DEV bool metal_finish(const DMaterial& m, D3 d_in, D3 n, D3 rs, D3& dir, F3& att) {
    const D3 reflected = reflect(unit(d_in), n);
    dir = reflected + m.fuzz_or_ir * rs; // the draw happens even when fuzz == 0
    att = mkf3(m.albedo[0], m.albedo[1], m.albedo[2]);
    return dot(dir, n) > 0.0;
}
template <bool FULLTEX = true>
RT_DEV bool isotropic_finish(const DeviceScene& S, const DMaterial& m, D3 p, double u, double v, D3 rs, D3& dir, F3& att, const PerlinTable* perlin0 = nullptr) {
    dir = rs; // not normalised (hit.rs:1007)
    att = tex_value<FULLTEX>(S, m.tex, u, v, p, perlin0);
    return true;
}
template <bool FULLTEX = true, class G>
RT_DEV bool scatter_lambertian(const DeviceScene& S, const DMaterial& m, D3 p, D3 n, double u, double v, G& g, D3& dir, F3& att,
                               const PerlinTable* perlin0 = nullptr) {
    g.begin_event();
    return lambertian_finish<FULLTEX>(S, m, p, n, u, v, random_in_unit_sphere(g), dir, att, perlin0);
}
template <class G> RT_DEV bool scatter_metal(const DMaterial& m, D3 d_in, D3 n, G& g, D3& dir, F3& att) {
    g.begin_event();
    return metal_finish(m, d_in, n, random_in_unit_sphere(g), dir, att);
}
RT_DEV double reflectance(double cosine, double ref_idx) { // hit.rs:1095-1099
    double r0 = (1.0 - ref_idx) / (1.0 + ref_idx);
    r0 = r0 * r0;
    const double x = 1.0 - cosine;
    return r0 + (1.0 - r0) * (x * x * x * x * x);
}
template <class G> RT_DEV bool scatter_dielectric(const DMaterial& m, D3 d_in, D3 n, bool front, G& g, D3& dir, F3& att) {
    g.begin_event();
    att = mkf3(1.f, 1.f, 1.f);
    const double ratio = front ? 1.0 / m.fuzz_or_ir : m.fuzz_or_ir;
    const D3 ud = unit(d_in);
    const double cos_theta = fmin(dot(-ud, n), 1.0);
    const double sin_theta = sqrt(1.0 - cos_theta * cos_theta);
    const bool cannot_refract = ratio * sin_theta > 1.0;
    if (cannot_refract || reflectance(cos_theta, ratio) > g.gen()) dir = reflect(ud, n); // `||` short-circuit: draw only if refraction is possible
    else dir = refract(ud, n, ratio);
    return true;
}
template <bool FULLTEX = true, class G>
RT_DEV bool scatter_isotropic(const DeviceScene& S, const DMaterial& m, D3 p, double u, double v, G& g, D3& dir, F3& att,
                              const PerlinTable* perlin0 = nullptr) {
    g.begin_event();
    return isotropic_finish<FULLTEX>(S, m, p, u, v, random_in_unit_sphere(g), dir, att, perlin0);
}

// ------------------------------------------------------------------ Camera::get_ray (camera.rs:59-71)
template <class G> RT_DEV Ray camera_get_ray(const DCamera& c, double s, double t, G& g) {
    double rx, ry;
    for (;;) { // random_in_unit_disk, vec3.rs:310-322 (runs even when lens_radius == 0)
        g.next2_pm1(rx, ry);
        if (rx * rx + ry * ry + 0.0 < 1.0) break;
    }
    rx *= c.lens_radius; ry *= c.lens_radius;
    const D3 u = mk3(c.u[0], c.u[1], c.u[2]), v = mk3(c.v[0], c.v[1], c.v[2]);
    const D3 offset = u * rx + v * ry;
    const D3 origin = mk3(c.origin[0], c.origin[1], c.origin[2]);
    const D3 llc = mk3(c.lower_left_corner[0], c.lower_left_corner[1], c.lower_left_corner[2]);
    const D3 hor = mk3(c.horizontal[0], c.horizontal[1], c.horizontal[2]), ver = mk3(c.vertical[0], c.vertical[1], c.vertical[2]);
    Ray r;
    r.o = origin + offset;
    r.d = llc + s * hor + t * ver - origin - offset;
    r.time = g.gen_range(c.time1, c.time2);
    return r;
}

// The first ray of a path: pixel jitter (world.rs:1212-1213), then Camera::get_ray (lens disk, shutter time).
template <class G> RT_DEV Ray camera_first_ray(const DCamera& c, int32_t ii, int32_t j, int32_t W, int32_t H, uint64_t seed, uint64_t path_id, uint32_t& draw_out) {
    G g;
    g.init(seed, path_id, 0);
    const double s = ((double)ii + g.gen()) / (double)(W - 1);
    const double t = ((double)j + g.gen()) / (double)(H - 1);
    const Ray r = camera_get_ray(c, s, t, g);
    draw_out = g.draw;
    return r;
}

} // namespace rtb
