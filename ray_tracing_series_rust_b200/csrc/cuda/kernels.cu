// kernels.cu — the wavefront path tracer (sm_100a).
//
// Replaces the reference's per-pixel hot loop (src/world.rs:1208-1216 -> Camera::get_ray ->
// ray_color world.rs:52-93 -> Hittable::hit / Material::scatter / Texture::value) with a pool of
// N resident path slots advanced one segment per iteration:
//
//   k_shade_all  (regeneration part) new camera rays: pixel jitter + Camera::get_ray, Philox    [a1,a2,a23]
//   k_extend     every live slot: world.hit(ray, 0.001, inf) incl. instances and media;
//                miss -> background * throughput into the pixel; hit -> HitRecord into the slot and the
//                slot index into the queue of its material type (warp-aggregated push)      [a3-a15]
//   k_shade<M>   one launch per material type over its queue: scatter / emitted, throughput update,
//                terminated paths add their radiance to the pixel and go to the newpath queue [a16-a22]
//
// Pixels accumulate in int64 fixed point (2^32 scale) with integer atomics: addition is associative,
// so the image is bit-reproducible for a given seed, independent of scheduling, slot count and of
// how the samples are sharded across GPUs.
#include "kernels.h"

#include <algorithm>
#include <cstdio>
#include <vector>

#ifndef RT_SHADE_MIN_BLOCKS
#define RT_SHADE_MIN_BLOCKS 3 // 80 registers, no spills: +1 % over 4 (64 registers, 204 B of spills) on Cornell smoke and book-2 final; 5 loses 2 %
#endif

#include "rt_device.cuh"

namespace rtb {

// ------------------------------------------------------------------ path state (SoA, one entry per slot)
// Four 32-byte chunks per slot, each in its own array: every access moves whole 32 B sectors with two
// 128-bit loads/stores, also when the slot indices come scattered out of a material queue.
struct alignas(32) SlotA { double ox, oy, oz, time; };                                   // ray origin (after a hit: HitRecord.p) + time
struct alignas(32) SlotB { double dx, dy, dz; uint32_t pad0, pad1; };                     // ray direction; for uv-reading materials (dx,dy) := (u,v) after the hit
struct alignas(32) SlotC { double nx, ny, nz; uint32_t hmat, pad; };                      // HitRecord.normal, material id | front_face << 31
struct alignas(32) SlotD { float tr, tg, tb; uint32_t draw; uint64_t path_id; uint32_t segment, pixel; }; // throughput, Philox stream + counter, ray_color iteration, pixel
struct PathState {
    SlotA* A;
    SlotB* B;
    SlotC* C;
    SlotD* D;
    uint8_t* alive;
};

// Queues: one per material type plus the miss queue.  Counts are double buffered by iteration parity:
// k_extend(i) fills counts[p], k_shade_all(i+1) drains counts[p] and clears counts[p^1].
#define Q_MISS MAT_TYPE_COUNT
#define Q_COUNT (MAT_TYPE_COUNT + 1)
struct Queues {
    uint32_t* q[Q_COUNT];
    uint32_t* counts;            // [2][8]
    uint32_t* dead;              // slots that found no more work
    uint32_t* ext_cursor;        // k_extend_p: next slot to hand out (reset by k_shade_all)
    unsigned long long* next_path;
    unsigned long long* stats;   // [0] segments, [1] nodes, [2] prims, [3] medium queries, [4..8] scatters by material
};

struct JobDev {
    int32_t W, H, rows, spp_total, sample_begin, max_depth;
    uint32_t npix_rendered;
    unsigned long long total_paths;
    uint64_t seed;
    uint32_t n_slots;
    int32_t count_events;
    uint32_t wait_thresh; // k_mega_r: finished lanes that end a traversal round
    uint32_t tile_rank, tile_count; // RT_RENDER_TILE_SHARD: npix_rendered counts this shard's pixels only; tile_count 0 = a pixel list
    uint32_t chunk;                 // fused kernels: consecutive path indices a warp claims per atomic
    unsigned long long path_base;   // this call renders the path indices [path_base, path_base + total_paths) of the sample-major enumeration
    const uint32_t* pix_list;       // rt_render_adaptive: dense index -> pixel of the active list (npix_rendered entries); null = no list
};

// Path-state chunks are streamed (read once / written once per kernel): evict-first hints keep them from
// pushing the BVH nodes and primitives out of L1 / L2.
template <class T> RT_DEV T ld_stream(const T* p) {
    static_assert(sizeof(T) == 32, "32-byte chunk");
    union { T t; uint4 q[2]; } u;
    u.q[0] = __ldcs(reinterpret_cast<const uint4*>(p));
    u.q[1] = __ldcs(reinterpret_cast<const uint4*>(p) + 1);
    return u.t;
}
template <class T> RT_DEV void st_stream(T* p, const T& v) {
    static_assert(sizeof(T) == 32, "32-byte chunk");
    union { T t; uint4 q[2]; } u;
    u.t = v;
    __stcs(reinterpret_cast<uint4*>(p), u.q[0]);
    __stcs(reinterpret_cast<uint4*>(p) + 1, u.q[1]);
}

RT_DEV uint32_t lane_id() { return threadIdx.x & 31u; }

// warp-aggregated queue push: lanes of the warp that push to the same counter share one atomic
RT_DEV uint32_t agg_reserve(uint32_t* counters, uint32_t key) {
    const unsigned act = __activemask();
    const unsigned grp = __match_any_sync(act, key);
    const int leader = __ffs(grp) - 1;
    const uint32_t rank = __popc(grp & ((1u << lane_id()) - 1u));
    uint32_t base = 0;
    if ((int)lane_id() == leader) base = atomicAdd(counters + key, (uint32_t)__popc(grp));
    base = __shfl_sync(grp, base, leader);
    return base + rank;
}

RT_DEV void accumulate(int64_t* __restrict__ accum, uint32_t pixel, float r, float g, float b) {
    // fixed point 2^32 in an int64 (2^31 units of headroom per channel); one sample is clamped to [0, 2^20]
    const double s = 4294967296.0;
    const double lim = 1048576.0;
    double v[3] = {(double)r, (double)g, (double)b};
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        double x = v[c];
        if (!(x > 0.0)) continue; // 0, negative, NaN contribute nothing
        x = x > lim ? lim : x;
        atomicAdd(reinterpret_cast<unsigned long long*>(accum + (size_t)pixel * 3 + c), (unsigned long long)(long long)(x * s + 0.5));
    }
}

// ------------------------------------------------------------------ k_init: every slot starts as a "miss" with zero throughput,
// so that the first k_shade_all launch does nothing but generate the first camera rays.
__global__ void k_init(PathState P, Queues Q, uint32_t n) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        Q.q[Q_MISS][i] = i;
        SlotD d;
        d.tr = 0.f; d.tg = 0.f; d.tb = 0.f; d.draw = 0; d.path_id = 0; d.segment = 0; d.pixel = 0;
        P.D[i] = d;
        P.alive[i] = 1;
    }
    if (blockIdx.x == 0 && threadIdx.x < 16) Q.counts[threadIdx.x] = (threadIdx.x == Q_MISS) ? n : 0u;
    if (blockIdx.x == 0 && threadIdx.x == 0) { *Q.dead = 0; *Q.next_path = 0ull; *Q.ext_cursor = 0; }
    if (blockIdx.x == 0 && threadIdx.x < 9) Q.stats[threadIdx.x] = 0ull;
}

// Tile sharding: the shard's pixels are enumerated densely (local row lr = band lr / 4 of this rank, line lr % 4);
// the global pixel index (accumulator address, Philox path id) is that of the unsharded image.
// A pixel list (adaptive sampling, tile_count 0) maps the dense index through the list instead.  The whole image (tile_count 1)
// stays one compare, as before the list existed.
RT_DEV uint32_t shard_pixel(const JobDev& J, uint32_t q) {
    if (J.tile_count == 1u) return q;
    if (J.tile_count == 0u) return __ldg(J.pix_list + q);
    const uint32_t W = (uint32_t)J.W, lr = q / W, x = q - lr * W;
    const uint32_t band = (lr / RT_TILE_ROWS) * J.tile_count + J.tile_rank;
    return (band * RT_TILE_ROWS + lr % RT_TILE_ROWS) * W + x;
}
// L -> (sample, pixel) without 64-bit integer division: quotient estimate in f64 (exact for L < 2^53) + one correction step
RT_DEV void split_path_index(unsigned long long L, uint32_t npix, uint32_t& s_local, uint32_t& pix) {
    uint32_t q = (uint32_t)__double2uint_rz(__ull2double_rz(L) / (double)npix);
    long long r = (long long)L - (long long)q * (long long)npix;
    if (r < 0) { --q; r += npix; }
    else if (r >= (long long)npix) { ++q; r -= npix; }
    s_local = q;
    pix = (uint32_t)r;
}

// Chunk claim of the persistent kernels (lane 0 of the warp): J.chunk consecutive path indices while much work is left, fewer towards
// the end (remaining / (2 x resident warps), at least 32), so that the warps run out of work within tens of microseconds of each other
// instead of one chunk time (512 paths = 0.6 ms on book-1: a fixed cost that an 11 ms strong-scaling shard feels).
RT_DEV unsigned long long claim_chunk(const JobDev& J, const Queues& Q, uint32_t& got) {
    const unsigned long long seen = *reinterpret_cast<volatile unsigned long long*>(Q.next_path);
    const unsigned long long rem = seen < J.total_paths ? J.total_paths - seen : 0ull;
    unsigned long long c = rem / (148ull * 7ull * 4ull * 2ull);
    c = c > (unsigned long long)J.chunk ? (unsigned long long)J.chunk : (c < 32ull ? 32ull : (c & ~31ull));
    got = (uint32_t)c;
    return atomicAdd(Q.next_path, c);
}

// New camera path into `slot` (pixel jitter world.rs:1212-1213 + Camera::get_ray), or retire the slot.
RT_DEV void regenerate(const DeviceScene& S, const JobDev& J, PathState& P, Queues& Q, uint32_t slot) {
    const unsigned act = __activemask();
    const int leader = __ffs(act) - 1;
    unsigned long long base = 0;
    if ((int)lane_id() == leader) base = atomicAdd(Q.next_path, (unsigned long long)__popc(act));
    base = __shfl_sync(act, base, leader);
    const unsigned long long L = base + __popc(act & ((1u << lane_id()) - 1u));
    if (L >= J.total_paths) {
        P.alive[slot] = 0;
        atomicAdd(Q.dead, 1u);
        return;
    }
    // sample-major order: consecutive path indices are neighbouring pixels of one sample => coherent primary rays
    uint32_t s_local, pix;
    split_path_index(L + J.path_base, J.npix_rendered, s_local, pix);
    pix = shard_pixel(J, pix);
    const int32_t j = (int32_t)(pix / (uint32_t)J.W), ii = (int32_t)(pix - (uint32_t)j * (uint32_t)J.W);
    const uint64_t path_id = (uint64_t)pix * (uint64_t)J.spp_total + (uint64_t)(J.sample_begin + (int32_t)s_local);
    uint32_t draw0;
    const Ray r = camera_first_ray<PathRng>(S.cam, ii, j, J.W, J.H, J.seed, path_id, draw0); // world.rs:1212-1214
    SlotA a; a.ox = r.o.x; a.oy = r.o.y; a.oz = r.o.z; a.time = r.time;
    SlotB b; b.dx = r.d.x; b.dy = r.d.y; b.dz = r.d.z; b.pad0 = 0; b.pad1 = 0;
    SlotD d; d.tr = 1.f; d.tg = 1.f; d.tb = 1.f; d.draw = draw0; d.path_id = path_id; d.segment = 0; d.pixel = pix;
    P.A[slot] = a;
    P.B[slot] = b;
    P.D[slot] = d;
}

// ------------------------------------------------------------------ k_extend: world.hit(ray, 0.001, inf) for every live slot
// WIDE = true: the main world is walked through its 4-wide collapse (DeviceScene::nodes4, Instance::root4)
template <bool MEDIA, bool COUNT, int MINB, bool GENERAL_MEDIA, uint32_t PM = RT_PM_ALL, bool WIDE = false>
__global__ void __launch_bounds__(128, MINB) k_extend(const __grid_constant__ DeviceScene S, const __grid_constant__ JobDev J, PathState P, Queues Q, int parity) {
    uint32_t* counts = Q.counts + 8 * parity;
    uint32_t my_segments = 0;
    TraceCounters tc; tc.nodes = 0; tc.prims = 0;
    for (uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x; slot < J.n_slots; slot += gridDim.x * blockDim.x) {
        if (!P.alive[slot]) continue;
        const SlotA a = ld_stream(&P.A[slot]);
        const SlotB b = ld_stream(&P.B[slot]);
        Ray r;
        r.o = mk3(a.ox, a.oy, a.oz);
        r.d = mk3(b.dx, b.dy, b.dz);
        r.time = a.time;
        uint64_t path_id = 0;
        uint32_t segment = 0;
        if (MEDIA) { const SlotD d = ld_stream(&P.D[slot]); path_id = d.path_id; segment = d.segment; }
        HitRec h;
        const bool hit = world_hit<COUNT, 2, MEDIA, GENERAL_MEDIA, PM, true, WIDE>(S, r, 0.001, RT_INF, true, J.seed, path_id, segment, h, &tc);
        ++my_segments;
        uint32_t qi = Q_MISS;
        if (hit) {
            SlotA na; na.ox = h.p.x; na.oy = h.p.y; na.oz = h.p.z; na.time = a.time;
            SlotC nc; nc.nx = h.n.x; nc.ny = h.n.y; nc.nz = h.n.z; nc.hmat = h.mat | (h.front ? 0x80000000u : 0u); nc.pad = 0;
            st_stream(&P.A[slot], na);
            st_stream(&P.C[slot], nc);
            const DMaterial* mp = &S.materials[h.mat];
            qi = __ldg(&mp->type);
            if (__ldg(&mp->flags) & 1u) { // the texture chain reads (u,v): such materials never read the incoming direction
                double2 uv = make_double2(h.u, h.v);
                *reinterpret_cast<double2*>(&P.B[slot]) = uv;
            }
        }
        Q.q[qi][agg_reserve(counts, qi)] = slot;
    }
    // statistics: one atomic per warp
    const unsigned full = 0xffffffffu;
    uint32_t segs = my_segments;
    for (int o = 16; o > 0; o >>= 1) segs += __shfl_xor_sync(full, segs, o);
    if (lane_id() == 0 && segs) atomicAdd(&Q.stats[0], (unsigned long long)segs);
    if (COUNT) {
        uint32_t a = tc.nodes, b = tc.prims;
        for (int o = 16; o > 0; o >>= 1) { a += __shfl_xor_sync(full, a, o); b += __shfl_xor_sync(full, b, o); }
        if (lane_id() == 0) { atomicAdd(&Q.stats[1], (unsigned long long)a); atomicAdd(&Q.stats[2], (unsigned long long)b); }
    }
}

// ------------------------------------------------------------------ k_extend_p: persistent, warp-scheduled world.hit
// Every lane owns one ray and is in one of three states; each turn the warp runs the phase that serves
// the most lanes per unit of cost (greedy), so lanes neither wait for the slowest lane's leaf search
// (while-while) nor for the longest ray of the warp (one ray per thread):
//   TRAV  one sibling-pair step of the BVH walk (64 B fetch, two f32 slab tests)
//   LEAF  the f64 primitive tests of the lane's pending leaves
//   ADV   traversal of the current instance finished: next instance, or media + HitRecord + queue push,
//         then fetch the next live slot (warp-aggregated claim of consecutive slots) and set it up
#ifndef RT_TRAV_STEPS
#define RT_TRAV_STEPS 3
#endif
#define RT_ST_TRAV 0
#define RT_ST_LEAF 1
#define RT_ST_ADV 2
#define RT_ST_EXIT 3
template <bool MEDIA, bool COUNT, int MINB>
__global__ void __launch_bounds__(128, MINB) k_extend_p(const __grid_constant__ DeviceScene S, const __grid_constant__ JobDev J, PathState P, Queues Q,
                                                         int parity) {
    uint32_t* counts = Q.counts + 8 * parity;
    const unsigned full = 0xffffffffu;
    const float4* __restrict__ nodes = reinterpret_cast<const float4*>(S.nodes);
    const bool planar = (S.flags & 1u) != 0;
    uint32_t stack[RT_STACK];
    int sp = 0;
    int state = RT_ST_ADV;
    bool have_ray = false;
    uint32_t slot = 0, inst_i = 0, cur = 0xffffffffu;
    uint32_t leaf_first0 = 0, leaf_cnt0 = 0, leaf_first1 = 0, leaf_cnt1 = 0;
    Ray r; // ray in the current instance's space
    r.o = mk3(0, 0, 0); r.d = mk3(0, 0, 1); r.time = 0.0;
    RayF f; f.idx = f.idy = f.idz = f.oodx = f.oody = f.oodz = 0.f;
    RayPre pre; pre.a = 1.0; pre.inv_a = 1.0; pre.inv_d = mk3(0, 0, 0);
    float tminf = 0.f, tmaxf = 0.f;
    BestHit best;
    best_init(best, RT_INF);
    uint32_t my_segments = 0;
    TraceCounters tc; tc.nodes = 0; tc.prims = 0;
    const uint32_t DONE = 0xffffffffu;
    const double t_min = 0.001;

    for (;;) {
        const unsigned mT = __ballot_sync(full, state == RT_ST_TRAV);
        const unsigned mL = __ballot_sync(full, state == RT_ST_LEAF);
        const unsigned mA = __ballot_sync(full, state == RT_ST_ADV);
        if (!(mT | mL | mA)) break;
        // greedy phase choice: lanes served per unit cost (pair step 1, leaf tests ~2.5, advance ~4)
        const int sT = __popc(mT) * 20, sL = __popc(mL) * 8, sA = __popc(mA) * 5;
        if (sT >= sL && sT >= sA) {
            // up to RT_TRAV_STEPS pair steps per scheduling decision (amortises the ballots)
            for (int step = 0; step < RT_TRAV_STEPS && state == RT_ST_TRAV; ++step) {
                const float4 lo0 = __ldg(nodes + 2 * cur), hi0 = __ldg(nodes + 2 * cur + 1);
                const float4 lo1 = __ldg(nodes + 2 * cur + 2), hi1 = __ldg(nodes + 2 * cur + 3);
                float tn0, tn1;
                bool h0 = slab(lo0, hi0, f, tminf, tmaxf, tn0);
                bool h1 = slab(lo1, hi1, f, tminf, tmaxf, tn1);
                if (COUNT) tc.nodes += 2;
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
                if ((leaf_cnt0 | leaf_cnt1) & 0xffffffu) state = RT_ST_LEAF;
                else { leaf_cnt0 = 0; leaf_cnt1 = 0; if (cur == DONE) state = RT_ST_ADV; }
            }
        } else if (sL >= sA) {
            if (state == RT_ST_LEAF) {
                for (int k = 0; k < 2; ++k) {
                    const uint32_t lc = k ? leaf_cnt1 : leaf_cnt0, lf = k ? leaf_first1 : leaf_first0;
                    if (lc & 0xffffffu) {
                        if (COUNT) tc.prims += lc & 0xffffffu;
                        leaf_test(S, r, pre, t_min, best, lc >> 24, lf, lc & 0xffffffu, inst_i);
                    }
                }
                leaf_cnt0 = 0; leaf_cnt1 = 0;
                tmaxf = f32_up(best.t);
                state = (cur == DONE) ? RT_ST_ADV : RT_ST_TRAV;
            }
        } else {
            if (state == RT_ST_ADV) {
                bool need_setup = false;
                if (have_ray) {
                    ++inst_i;
                    if (inst_i < S.n_main_instances) {
                        need_setup = true;
                    } else {
                        // world.hit is complete for this ray: media, HitRecord, queue push
                        const SlotA a = P.A[slot];
                        const SlotB b = P.B[slot];
                        Ray wr;
                        wr.o = mk3(a.ox, a.oy, a.oz); wr.d = mk3(b.dx, b.dy, b.dz); wr.time = a.time;
                        HitRec h;
                        bool hit = false;
                        if (MEDIA) {
                            const SlotD d = P.D[slot];
                            double closest = best.t;
                            int32_t mwin = -1;
                            D3 mp = mk3(0, 0, 0);
                            for (uint32_t mi = 0; mi < S.n_media; ++mi) medium_query<COUNT, false>(S, mi, wr, t_min, closest, mwin, mp, J.seed, d.path_id, d.segment, &tc);
                            if (mwin >= 0) {
                                const Medium md = S.media[mwin];
                                h.p = mp; h.n = mk3(0, 0, 0); h.t = closest; h.u = 0.0; h.v = 0.0; h.front = true; // hit.rs:975-984
                                h.mat = md.mat_id; h.prim_id = md.prim_id;
                                hit = true;
                            }
                        }
                        if (!hit && best.type != RT_NONE) { h = finalize_hit<2>(S, wr, best); hit = true; }
                        uint32_t qi = Q_MISS;
                        if (hit) {
                            SlotA na; na.ox = h.p.x; na.oy = h.p.y; na.oz = h.p.z; na.time = a.time;
                            SlotC nc; nc.nx = h.n.x; nc.ny = h.n.y; nc.nz = h.n.z; nc.hmat = h.mat | (h.front ? 0x80000000u : 0u); nc.pad = 0;
                            P.A[slot] = na;
                            P.C[slot] = nc;
                            const DMaterial* mp2 = &S.materials[h.mat];
                            qi = __ldg(&mp2->type);
                            if (__ldg(&mp2->flags) & 1u) *reinterpret_cast<double2*>(&P.B[slot]) = make_double2(h.u, h.v);
                        }
                        Q.q[qi][agg_reserve(counts, qi)] = slot;
                        have_ray = false;
                    }
                }
                if (!have_ray) {
                    // claim the next slot (consecutive slots for the lanes fetching together => coalesced state loads)
                    const unsigned act = __activemask();
                    const int leader = __ffs(act) - 1;
                    uint32_t base = 0;
                    if ((int)lane_id() == leader) base = atomicAdd(Q.ext_cursor, (uint32_t)__popc(act));
                    base = __shfl_sync(act, base, leader);
                    slot = base + __popc(act & ((1u << lane_id()) - 1u));
                    if (slot >= J.n_slots) {
                        state = RT_ST_EXIT;
                    } else if (P.alive[slot]) {
                        have_ray = true;
                        inst_i = 0;
                        best_init(best, RT_INF);
                        ++my_segments;
                        need_setup = true;
                    } // dead slot: stay in ADV and fetch again
                }
                if (need_setup) {
                    const SlotA a = P.A[slot];
                    const SlotB b = P.B[slot];
                    r.o = mk3(a.ox, a.oy, a.oz); r.d = mk3(b.dx, b.dy, b.dz); r.time = a.time;
                    const Instance* ip = &S.instances[inst_i];
                    xform_ray(S.ops, __ldg(&ip->chain_off), __ldg(&ip->chain_len), r);
                    f = make_rayf(r);
                    pre = make_raypre(r, planar);
                    tminf = f32_down(t_min);
                    tmaxf = f32_up(best.t);
                    cur = __ldg(&ip->root);
                    sp = 0;
                    leaf_cnt0 = 0; leaf_cnt1 = 0;
                    state = RT_ST_TRAV;
                }
            }
        }
    }
    uint32_t segs = my_segments;
    for (int o = 16; o > 0; o >>= 1) segs += __shfl_xor_sync(full, segs, o);
    if (lane_id() == 0 && segs) atomicAdd(&Q.stats[0], (unsigned long long)segs);
    if (COUNT) {
        uint32_t a = tc.nodes, b = tc.prims;
        for (int o = 16; o > 0; o >>= 1) { a += __shfl_xor_sync(full, a, o); b += __shfl_xor_sync(full, b, o); }
        if (lane_id() == 0) { atomicAdd(&Q.stats[1], (unsigned long long)a); atomicAdd(&Q.stats[2], (unsigned long long)b); }
    }
}

// ------------------------------------------------------------------ k_shade_all: one launch drains every material queue and the miss queue.
// The flat work index space is the concatenation of the queues, each padded to a multiple of 32, so a
// warp only ever holds entries of ONE queue (material-coherent warps without one launch per material).
// Paths that end here (miss, light, absorbed, depth exhausted) add their radiance to the pixel and the
// slot is refilled in place with the next camera path.
__global__ void __launch_bounds__(256, RT_SHADE_MIN_BLOCKS) k_shade_all(const __grid_constant__ DeviceScene S, const __grid_constant__ JobDev J, PathState P, Queues Q,
                                                   int64_t* __restrict__ accum, int parity) {
    // perlin.rs tables of the scene's first Noise texture staged in shared memory (6.9 KB: 256 f64 gradients + 3 x 256 byte
    // permutations): the 7-octave turbulence gathers 8 x 7 = 56 gradients per shaded point from here instead of L1 / L2
    __shared__ PerlinTable s_perlin;
    const bool stage_perlin = (S.flags & 8u) != 0;
    if (stage_perlin) {
        const uint4* src = reinterpret_cast<const uint4*>(S.perlin);
        uint4* dst = reinterpret_cast<uint4*>(&s_perlin);
        for (uint32_t i = threadIdx.x; i < sizeof(PerlinTable) / 16; i += blockDim.x) dst[i] = __ldg(src + i);
        __syncthreads();
    }
    const PerlinTable* perlin0 = stage_perlin ? &s_perlin : nullptr;
    const uint32_t* counts = Q.counts + 8 * parity;
    uint32_t start[Q_COUNT + 1];
    start[0] = 0;
#pragma unroll
    for (int q = 0; q < Q_COUNT; ++q) start[q + 1] = start[q] + ((counts[q] + 31u) & ~31u);
    const uint32_t total = start[Q_COUNT];
    if (blockIdx.x == 0 && threadIdx.x < 8) {
        Q.counts[8 * (parity ^ 1) + threadIdx.x] = 0; // next k_extend fills the other buffer
        if (threadIdx.x == 0) *Q.ext_cursor = 0;
        if (threadIdx.x < MAT_TYPE_COUNT && counts[threadIdx.x]) atomicAdd(&Q.stats[4 + threadIdx.x], (unsigned long long)counts[threadIdx.x]);
    }
    for (uint32_t f = blockIdx.x * blockDim.x + threadIdx.x; f < total; f += gridDim.x * blockDim.x) {
        int q = 0;
#pragma unroll
        for (int k = 1; k < Q_COUNT; ++k) q += (f >= start[k]) ? 1 : 0;
        const uint32_t i = f - start[q];
        if (i >= counts[q]) continue; // padding lane
        const uint32_t slot = Q.q[q][i];
        SlotD sd = P.D[slot];
        F3 contrib = mkf3(0.f, 0.f, 0.f);
        bool ended = true;
        if (q == Q_MISS) {
            // world.rs:86-89: output += product * background
            F3 bg = mkf3(S.background[0], S.background[1], S.background[2]);
            if (S.bg_gradient) { const SlotB sb = P.B[slot]; bg = miss_color(S, mk3(sb.dx, sb.dy, sb.dz)); } // a miss leaves the ray direction in B
            contrib = mkf3(sd.tr * bg.x, sd.tg * bg.y, sd.tb * bg.z);
        } else {
            const SlotA sa = P.A[slot];
            const SlotC sc = P.C[slot];
            const uint32_t hm = sc.hmat;
            const DMaterial m = S.materials[hm & 0x7fffffffu];
            const D3 p = mk3(sa.ox, sa.oy, sa.oz);
            double hu = 0.0, hv = 0.0;
            D3 d_in = mk3(0, 0, 0);
            if (q == MAT_METAL || q == MAT_DIELECTRIC) {
                const SlotB sb = P.B[slot];
                d_in = mk3(sb.dx, sb.dy, sb.dz);
            } else if (m.flags & 1u) {
                const double2 uv = *reinterpret_cast<const double2*>(&P.B[slot]);
                hu = uv.x; hv = uv.y;
            }
            if (q == MAT_LIGHT) {
                const F3 e = tex_value(S, m.tex, hu, hv, p, perlin0); // hit.rs:1146-1151, world.rs:78-84
                contrib = mkf3(sd.tr * e.x, sd.tg * e.y, sd.tb * e.z);
            } else {
                PathRng g;
                g.init(J.seed, sd.path_id, sd.draw);
                const D3 n3 = mk3(sc.nx, sc.ny, sc.nz);
                D3 dir = mk3(0, 0, 0);
                F3 att = mkf3(0.f, 0.f, 0.f);
                bool scattered;
                if (q == MAT_LAMBERTIAN) scattered = scatter_lambertian(S, m, p, n3, hu, hv, g, dir, att, perlin0);
                else if (q == MAT_METAL) scattered = scatter_metal(m, d_in, n3, g, dir, att);
                else if (q == MAT_DIELECTRIC) scattered = scatter_dielectric(m, d_in, n3, (hm >> 31) != 0, g, dir, att);
                else scattered = scatter_isotropic(S, m, p, hu, hv, g, dir, att, perlin0);
                const uint32_t seg = sd.segment + 1;
                if (scattered && (int32_t)seg < J.max_depth) { // world.rs:64-67: at most max_depth hit queries per path
                    sd.tr *= att.x; sd.tg *= att.y; sd.tb *= att.z; // world.rs:75
                    sd.draw = g.draw;
                    sd.segment = seg;
                    SlotB nb; nb.dx = dir.x; nb.dy = dir.y; nb.dz = dir.z; nb.pad0 = 0; nb.pad1 = 0; // the origin already is rec.p
                    P.B[slot] = nb;
                    P.D[slot] = sd;
                    ended = false;
                }
                // absorbed (Metal) or depth exhausted: the path keeps what it has (nothing: emitters do not scatter)
            }
        }
        if (ended) {
            accumulate(accum, sd.pixel, contrib.x, contrib.y, contrib.z);
            regenerate(S, J, P, Q, slot);
        }
    }
}

// ------------------------------------------------------------------ k_mega: persistent fused variant (RT_MODE_FUSED)
// One thread owns one path at a time and keeps its whole state in registers: generate -> world.hit ->
// scatter -> ... until the path ends, then the lane pulls the next path index.  No path state and no
// queues in HBM, one launch per render.  Path indices are claimed per warp in chunks of CHUNK
// consecutive indices (= neighbouring pixels of one sample), so a warp's primary rays stay spatially
// close.  Same device functions, same Philox streams, same integer accumulation as the wavefront: the
// two modes produce bit-identical images.
#define RT_MEGA_CHUNK 512u // path indices a warp claims at once; the host lowers it (JobDev.chunk) for short renders, see launch_render
// WIDE = true (media-free, wrapper-free, single instance): world.hit walks the 4-wide collapse (DeviceScene::nodes4).
#ifndef RT_CAM_BATCH
#define RT_CAM_BATCH 1
#endif
// Camera rays are generated 32 at a time by the whole warp into a per-warp buffer in shared memory, and ended lanes take theirs from
// it: pixel jitter, lens-disk rejection loop and the two Philox blocks of a new path run at 32 lanes every third iteration or so
// instead of at the ~10 lanes that happen to have ended in this one.  Measured: book-1 final 70.3 -> 68.2 ms (profiles/r2_57_ab_cam_batch.txt);
// on the sibling-pair kernels of the moving / gravity sphere scenes +-0 / -2.2 % (their walks miss the 9 KB per CTA that the buffer
// takes from L1), on the same scenes' 4-wide kernels +5.4 % / +0.2 % (r2_67): the three sphere kernels on the 4-wide tree use it
// (RT_CAM_BATCH = 0: none does).  The buffer (8.6 KB per CTA) also holds the warps' refill state.
template <bool ON> struct CamBufferT {
    double v[4][7][32]; // [warp][o.x o.y o.z d.x d.y d.z time][entry]
    uint32_t sample[4][32], pixel[4][32], draw[4][32];
    // The warp-uniform refill state: read and written once per refill, so it lives here rather than in 7 registers of every lane for
    // the whole kernel (part of what fits the kernel into 80 registers, 6 CTAs/SM)
    unsigned long long chunk_next[4], chunk_end[4];
    uint32_t head[4], count[4], gen_done[4]; // gen_done: the path indices have run out
    uint32_t dry[4];                         // gen_done and the buffer is empty: idle lanes of the warp stay idle
};
template <> struct CamBufferT<false> {};
// What a lane keeps of its path besides the ray: read and written in the shading code only, never in the walk.  The camera-batch kernels
// keep it in shared memory ([thread], 9 words: an odd stride, conflict free), so that it takes no registers while the lane walks the tree.
struct PathVars {
    float tr, tg, tb;             // throughput (world.rs:57 `product`)
    uint32_t pixel, sample, draw; // the path id pixel * spp_total + sample is formed where Philox needs it; Philox draw counter
    uint32_t segment, segs, pad;  // ray_color iteration; segments this lane has traced (statistics)
};
template <bool SMEM> struct PathVarsT {};
template <> struct PathVarsT<true> { PathVars v[128]; };
template <bool SMEM> RT_DEV PathVars& path_vars(PathVarsT<SMEM>& sm, PathVars& reg) {
    if constexpr (SMEM) return sm.v[threadIdx.x];
    else return reg;
}
// FULLTEX = false: the scene has no Noise and no Image texture (DeviceScene::flags bits 3 and 4 clear): the Perlin and texel code and the
// sphere (u, v) are compiled out.  The Perlin turbulence is the register peak of the kernel (tools/reg_pressure.py: 93 live at 5 CTAs/SM).
template <bool MEDIA, int MINB, bool GENERAL_MEDIA, uint32_t PM = RT_PM_ALL, bool XF = true, bool WIDE = false, bool FULLTEX = true>
__global__ void __launch_bounds__(128, MINB) k_mega(const __grid_constant__ DeviceScene S, const __grid_constant__ JobDev J, Queues Q,
                                                      int64_t* __restrict__ accum) {
    const unsigned full = 0xffffffffu;
    unsigned long long chunk_next = 0, chunk_end = 0; // warp-uniform (the camera-batch kernels keep theirs in CamBufferT)
    Ray r;
    r.o = mk3(0, 0, 0); r.d = mk3(0, 0, 1); r.time = 0.0;
    bool alive = false, exhausted = false;
    constexpr bool CAMB = RT_CAM_BATCH && WIDE && (PM == 0x1u || PM == 0x3u || PM == 0x5u);
    __shared__ CamBufferT<CAMB> cam;
    __shared__ PathVarsT<CAMB> pv_smem;
    PathVars pv_reg;
    PathVars& pv = path_vars<CAMB>(pv_smem, pv_reg);
    pv.tr = pv.tg = pv.tb = 0.f;
    pv.pixel = 0; pv.sample = 0; pv.draw = 0; pv.segment = 0; pv.segs = 0;
    const uint32_t wid = threadIdx.x >> 5, ln = lane_id();
    if constexpr (CAMB) {
        if (ln == 0) { cam.chunk_next[wid] = 0; cam.chunk_end[wid] = 0; cam.head[wid] = 0; cam.count[wid] = 0; cam.gen_done[wid] = 0; cam.dry[wid] = 0; }
        __syncwarp();
    }
    for (;;) {
        // ---- refill idle lanes
        bool idle = !alive; // and not out of work: `exhausted`, which the camera-batch kernels keep per warp (dry) instead of per lane
        if constexpr (CAMB) idle = idle && cam.dry[wid] == 0u;
        else idle = idle && !exhausted;
        const unsigned need = __ballot_sync(full, idle);
        if constexpr (CAMB) {
          if (need) {
            uint32_t buf_head = cam.head[wid], buf_count = cam.count[wid];
            bool gen_done = cam.gen_done[wid] != 0;
            uint32_t rank = __popc(need & ((1u << ln) - 1u));
            bool want = idle;
            for (int round = 0; round < 2; ++round) { // what the buffer holds first; then, if lanes are left over, 32 new rays and the rest
                const uint32_t want_n = __popc(__ballot_sync(full, want));
                const uint32_t served = want_n < buf_count ? want_n : buf_count;
                if (want && rank < served) {
                    const uint32_t e = buf_head + rank;
                    r.o = mk3(cam.v[wid][0][e], cam.v[wid][1][e], cam.v[wid][2][e]);
                    r.d = mk3(cam.v[wid][3][e], cam.v[wid][4][e], cam.v[wid][5][e]);
                    r.time = cam.v[wid][6][e];
                    pv.sample = cam.sample[wid][e]; pv.pixel = cam.pixel[wid][e]; pv.draw = cam.draw[wid][e];
                    pv.tr = pv.tg = pv.tb = 1.f;
                    pv.segment = 0;
                    alive = true;
                    want = false;
                } else if (want) {
                    rank -= served;
                }
                buf_head += served; buf_count -= served;
                if (served == want_n) break;
                if (round == 1 || gen_done) break; // lanes still wanting are out of work: the buffer is empty and gen_done is set
                // the buffer is empty: the whole warp generates the next 32 camera rays
                __syncwarp();
                unsigned long long c_next = cam.chunk_next[wid], c_end = cam.chunk_end[wid];
                if (c_next == c_end) {
                    unsigned long long base = 0;
                    uint32_t got = 0;
                    if (ln == 0) base = claim_chunk(J, Q, got);
                    base = __shfl_sync(full, base, 0);
                    got = __shfl_sync(full, got, 0);
                    c_next = base; c_end = base + got;
                }
                const unsigned long long L = c_next + ln;
                const bool valid = L < J.total_paths;
                if (valid) {
                    uint32_t s_local, pix, d0;
                    split_path_index(L + J.path_base, J.npix_rendered, s_local, pix);
                    pix = shard_pixel(J, pix);
                    const int32_t j = (int32_t)(pix / (uint32_t)J.W), ii = (int32_t)(pix - (uint32_t)j * (uint32_t)J.W);
                    const uint32_t smp = (uint32_t)(J.sample_begin + (int32_t)s_local);
                    const uint64_t pid = (uint64_t)pix * (uint64_t)J.spp_total + (uint64_t)smp;
                    const Ray cr = camera_first_ray<PathRngOol>(S.cam, ii, j, J.W, J.H, J.seed, pid, d0); // world.rs:1212-1214
                    cam.v[wid][0][ln] = cr.o.x; cam.v[wid][1][ln] = cr.o.y; cam.v[wid][2][ln] = cr.o.z;
                    cam.v[wid][3][ln] = cr.d.x; cam.v[wid][4][ln] = cr.d.y; cam.v[wid][5][ln] = cr.d.z;
                    cam.v[wid][6][ln] = cr.time;
                    cam.sample[wid][ln] = smp; cam.pixel[wid][ln] = pix; cam.draw[wid][ln] = d0;
                }
                buf_head = 0;
                buf_count = __popc(__ballot_sync(full, valid)); // valid lanes are a prefix: L grows with the lane
                if (buf_count < 32u) gen_done = true;
                __syncwarp();
                if (ln == 0) { cam.chunk_next[wid] = c_next + 32; cam.chunk_end[wid] = c_end; }
                __syncwarp();
            }
            __syncwarp();
            if (ln == 0) {
                cam.head[wid] = buf_head; cam.count[wid] = buf_count; cam.gen_done[wid] = gen_done ? 1u : 0u;
                cam.dry[wid] = (gen_done && buf_count == 0u) ? 1u : 0u;
            }
            __syncwarp();
          }
        } else if (need) {
            const uint32_t n_need = __popc(need);
            // make sure the warp's chunk covers the request; leftover indices of the old chunk are used first
            unsigned long long avail = chunk_end - chunk_next;
            unsigned long long second_base = 0;
            uint32_t got = 0;
            if (avail < n_need) {
                if (lane_id() == 0) second_base = claim_chunk(J, Q, got);
                second_base = __shfl_sync(full, second_base, 0);
                got = __shfl_sync(full, got, 0);
            }
            if (!alive && !exhausted) {
                const uint32_t rank = __popc(need & ((1u << lane_id()) - 1u));
                unsigned long long L = (rank < avail) ? chunk_next + rank : second_base + (rank - avail);
                if (L >= J.total_paths) {
                    exhausted = true;
                } else {
                    uint32_t s_local;
                    split_path_index(L + J.path_base, J.npix_rendered, s_local, pv.pixel);
                    pv.pixel = shard_pixel(J, pv.pixel);
                    const int32_t j = (int32_t)(pv.pixel / (uint32_t)J.W), ii = (int32_t)(pv.pixel - (uint32_t)j * (uint32_t)J.W);
                    pv.sample = (uint32_t)(J.sample_begin + (int32_t)s_local);
                    r = camera_first_ray<PathRngOol>(S.cam, ii, j, J.W, J.H, J.seed, (uint64_t)pv.pixel * (uint64_t)J.spp_total + (uint64_t)pv.sample, pv.draw); // world.rs:1212-1214
                    pv.tr = pv.tg = pv.tb = 1.f;
                    pv.segment = 0;
                    alive = true;
                }
            }
            if (avail < n_need) { chunk_next = second_base + (n_need - avail); chunk_end = second_base + got; }
            else chunk_next += n_need;
        }
        if (!__any_sync(full, alive)) break;
        if (!alive) continue;
        // ---- one ray_color iteration (world.rs:63-91)
        HitRec h;
        bool hit;
        if (WIDE) {
            BestHit best;
            best_init(best, RT_INF);
            unsigned long long wstack[RT_WIDE_STACK];
            uint32_t cur = S.root4;
            int sp = 0;
            trace_wide<PM, false>(S, r, 0.001, best, cur, sp, wstack, 0u);
            hit = best.type != RT_NONE;
            if (hit) h = finalize_hit<FULLTEX ? 2 : 0, PM, false>(S, r, best);
        } else {
            hit = world_hit<false, 2, MEDIA, GENERAL_MEDIA, PM, XF>(S, r, 0.001, RT_INF, true, J.seed, (uint64_t)pv.pixel * (uint64_t)J.spp_total + (uint64_t)pv.sample,
                                                                    pv.segment, h, nullptr);
        }
        ++pv.segs;
        F3 contrib = mkf3(0.f, 0.f, 0.f);
        bool ended = true;
        if (!hit) {
            const F3 bg = miss_color(S, r.d);
            contrib = mkf3(pv.tr * bg.x, pv.tg * bg.y, pv.tb * bg.z);
        } else {
            const DMaterial m = S.materials[h.mat];
            if (m.type == MAT_LIGHT) {
                const F3 e = tex_value<FULLTEX>(S, m.tex, h.u, h.v, h.p);
                contrib = mkf3(pv.tr * e.x, pv.tg * e.y, pv.tb * e.z);
            } else {
                PathRngOolBegun g;
                g.init(J.seed, (uint64_t)pv.pixel * (uint64_t)J.spp_total + (uint64_t)pv.sample, pv.draw);
                g.open_event(); // Material::scatter starts on a block boundary: the first block for every scattering lane at once
                D3 dir = mk3(0, 0, 0), rs = mk3(0, 0, 0);
                F3 att = mkf3(0.f, 0.f, 0.f);
                bool scattered;
                if (m.type != MAT_DIELECTRIC) rs = random_in_unit_sphere(g); // one rejection loop for Lambertian, Metal and Isotropic lanes
                if (m.type == MAT_LAMBERTIAN) scattered = lambertian_finish<FULLTEX>(S, m, h.p, h.n, h.u, h.v, rs, dir, att);
                else if (m.type == MAT_METAL) scattered = metal_finish(m, r.d, h.n, rs, dir, att);
                else if (m.type == MAT_DIELECTRIC) scattered = scatter_dielectric(m, r.d, h.n, h.front, g, dir, att);
                else scattered = isotropic_finish<FULLTEX>(S, m, h.p, h.u, h.v, rs, dir, att);
                if (scattered && (int32_t)(pv.segment + 1) < J.max_depth) {
                    pv.tr *= att.x; pv.tg *= att.y; pv.tb *= att.z;
                    r.o = h.p; r.d = dir;
                    pv.draw = g.draw;
                    ++pv.segment;
                    ended = false;
                }
            }
        }
        if (ended) {
            accumulate(accum, pv.pixel, contrib.x, contrib.y, contrib.z);
            alive = false;
        }
    }
    uint32_t segs = pv.segs;
    for (int o = 16; o > 0; o >>= 1) segs += __shfl_xor_sync(full, segs, o);
    if (lane_id() == 0 && segs) atomicAdd(&Q.stats[0], (unsigned long long)segs);
}

// k_mega_r: k_mega with the resumable traversal (single main instance, no wrappers, no media).  Each round:
// idle lanes claim new paths -> every lane with a ray walks the BVH until `wait_thresh` lanes have finished ->
// the finished lanes shade / scatter / start their next segment, the others keep their traversal state and
// continue in the next round.  Per-path arithmetic and Philox streams are those of k_mega: bit-identical images.
// WIDE = true walks the 4-wide collapse of the tree (DeviceScene::nodes4, trace_wide) instead of the sibling pairs.
template <int MINB, uint32_t PM, bool WIDE = false>
__global__ void __launch_bounds__(128, MINB) k_mega_r(const __grid_constant__ DeviceScene S, const __grid_constant__ JobDev J, Queues Q,
                                                        int64_t* __restrict__ accum) {
    const unsigned full = 0xffffffffu;
    const uint32_t DONE = 0xffffffffu;
    unsigned long long chunk_next = 0, chunk_end = 0; // warp-uniform
    Ray r;
    r.o = mk3(0, 0, 0); r.d = mk3(0, 0, 1); r.time = 0.0;
    float tr = 0.f, tg = 0.f, tb = 0.f;
    uint32_t pixel = 0, draw = 0, segment = 0;
    uint64_t path_id = 0;
    bool alive = false, exhausted = false;
    uint32_t my_segments = 0;
    uint32_t stack[WIDE ? 1 : RT_STACK];
    unsigned long long wstack[WIDE ? RT_WIDE_STACK : 1];
    uint32_t cur = DONE;
    int sp = 0;
    BestHit best;
    best_init(best, RT_INF);
    const uint32_t root = WIDE ? S.root4 : __ldg(&S.instances[0].root);
    for (;;) {
        // ---- refill idle lanes
        const unsigned need = __ballot_sync(full, !alive && !exhausted);
        if (need) {
            const uint32_t n_need = __popc(need);
            unsigned long long avail = chunk_end - chunk_next;
            unsigned long long second_base = 0;
            uint32_t got = 0;
            if (avail < n_need) {
                if (lane_id() == 0) second_base = claim_chunk(J, Q, got);
                second_base = __shfl_sync(full, second_base, 0);
                got = __shfl_sync(full, got, 0);
            }
            if (!alive && !exhausted) {
                const uint32_t rank = __popc(need & ((1u << lane_id()) - 1u));
                unsigned long long L = (rank < avail) ? chunk_next + rank : second_base + (rank - avail);
                if (L >= J.total_paths) {
                    exhausted = true;
                } else {
                    uint32_t s_local;
                    split_path_index(L + J.path_base, J.npix_rendered, s_local, pixel);
                    pixel = shard_pixel(J, pixel);
                    const int32_t j = (int32_t)(pixel / (uint32_t)J.W), ii = (int32_t)(pixel - (uint32_t)j * (uint32_t)J.W);
                    path_id = (uint64_t)pixel * (uint64_t)J.spp_total + (uint64_t)(J.sample_begin + (int32_t)s_local);
                    r = camera_first_ray<PathRngOol>(S.cam, ii, j, J.W, J.H, J.seed, path_id, draw); // world.rs:1212-1214
                    tr = tg = tb = 1.f;
                    segment = 0;
                    alive = true;
                    best_init(best, RT_INF);
                    cur = root; sp = 0;
                }
            }
            if (avail < n_need) { chunk_next = second_base + (n_need - avail); chunk_end = second_base + got; }
            else chunk_next += n_need;
        }
        if (!__any_sync(full, alive)) break;
        // ---- world.hit for every lane that has a ray; returns when enough lanes are ready to shade
        if (WIDE) trace_wide<PM, true>(S, r, 0.001, best, cur, sp, wstack, J.wait_thresh);
        else trace_resume<PM>(S, r, 0.001, best, cur, sp, stack, J.wait_thresh);
        if (!alive || cur != DONE) continue;
        // ---- the rest of this ray_color iteration (world.rs:63-91)
        ++my_segments;
        F3 contrib = mkf3(0.f, 0.f, 0.f);
        bool ended = true;
        if (best.type == RT_NONE) {
            const F3 bg = miss_color(S, r.d);
            contrib = mkf3(tr * bg.x, tg * bg.y, tb * bg.z);
        } else {
            const HitRec h = finalize_hit<2, PM, false>(S, r, best);
            const DMaterial m = S.materials[h.mat];
            if (m.type == MAT_LIGHT) {
                const F3 e = tex_value(S, m.tex, h.u, h.v, h.p);
                contrib = mkf3(tr * e.x, tg * e.y, tb * e.z);
            } else {
                PathRngOolBegun g;
                g.init(J.seed, path_id, draw);
                g.open_event(); // Material::scatter starts on a block boundary: the first block for every scattering lane at once
                D3 dir = mk3(0, 0, 0), rs = mk3(0, 0, 0);
                F3 att = mkf3(0.f, 0.f, 0.f);
                bool scattered;
                if (m.type != MAT_DIELECTRIC) rs = random_in_unit_sphere(g); // one rejection loop for Lambertian, Metal and Isotropic lanes
                if (m.type == MAT_LAMBERTIAN) scattered = lambertian_finish(S, m, h.p, h.n, h.u, h.v, rs, dir, att);
                else if (m.type == MAT_METAL) scattered = metal_finish(m, r.d, h.n, rs, dir, att);
                else if (m.type == MAT_DIELECTRIC) scattered = scatter_dielectric(m, r.d, h.n, h.front, g, dir, att);
                else scattered = isotropic_finish(S, m, h.p, h.u, h.v, rs, dir, att);
                if (scattered && (int32_t)(segment + 1) < J.max_depth) {
                    tr *= att.x; tg *= att.y; tb *= att.z;
                    r.o = h.p; r.d = dir;
                    draw = g.draw;
                    ++segment;
                    ended = false;
                    best_init(best, RT_INF);
                    cur = root; sp = 0;
                }
            }
        }
        if (ended) {
            accumulate(accum, pixel, contrib.x, contrib.y, contrib.z);
            alive = false;
        }
    }
    uint32_t segs = my_segments;
    for (int o = 16; o > 0; o >>= 1) segs += __shfl_xor_sync(full, segs, o);
    if (lane_id() == 0 && segs) atomicAdd(&Q.stats[0], (unsigned long long)segs);
}

// ------------------------------------------------------------------ k_pool: warp-local wavefront in shared memory (RT_MODE_POOL)
// k_mega keeps one path per lane in registers, so a warp's lanes wait for each other twice per segment: at the end of the BVH walk (the
// longest ray of 32 decides) and in the shading code (32 lanes, 3-4 materials, rejection loops) - ncu: 11.3 of 32 lanes active per
// instruction on book-1, 6.8 on the 871 200-triangle mesh.  The global wavefront (k_extend / k_shade_all) fixes the shading half with
// per-material queues but pays 300 B of path state per segment through HBM / L2 and still walks one ray per lane to the end.
// Here every WARP owns a pool of P paths in shared memory (~100 B of state per path) and small slot lists, all private to the warp (no
// block-level synchronisation, no atomics besides the pixel sums), and alternates three phases:
//   REGEN  ended slots get the next camera paths (pixel jitter + Camera::get_ray, world.rs:1212-1214) in full batches of 32
//   TRACE  world.hit (world.rs:68): a lane that finishes its walk stores (t, primitive) in the slot, takes the next waiting ray from the
//          list and goes on - the lanes stay busy as long as rays wait.  When the list runs dry and more than a quarter of the lanes
//          idle, the warp goes shading; the walks still in flight stay in their lanes' registers and resume in the next TRACE phase
//          (resumable walks as in k_mega_r), so no phase ever waits for its longest ray
//   SHADE  finished slots are classified (miss / light / Lambertian / Metal+Dielectric / Isotropic; media are sampled here, all lanes
//          together) into per-material lists, and each list is shaded in batches of 32: HitRecord rebuild + Material::scatter run
//          material-coherent; survivors go back to the TRACE list, ended paths add their radiance to the pixel and go to REGEN
// Per-path arithmetic, Philox streams and the integer pixel sums are those of the other two modes: the image is bit-identical.
#define RT_POOL_MISS 0xffffffffu
#define RT_POOL_IDX_BITS 26
template <int P>
struct alignas(16) WarpPool {
    double ox[P], oy[P], oz[P], dx[P], dy[P], dz[P], time[P]; // the ray of the slot's current segment, world space
    double best_t[P];                                        // closest_so_far of the finished world.hit
    uint32_t best_ref[P];                                    // RT_POOL_MISS | type << 29 | side << 26 | index (type PRIM_MEDIUM: index = medium)
    float tr[P], tg[P], tb[P];                               // throughput (world.rs:57 `product`)
    uint32_t pixel[P], s_local[P];                           // path id = pixel * spp_total + sample_begin + s_local
    uint32_t draw[P];                                        // Philox draw counter of the path
    uint8_t segment[P], best_inst[P];
    uint8_t q_trace[P], q_done[P], q_regen[P], q_mat[4][P];  // slot lists: waiting for world.hit / hit found / path ended / by material class
};
RT_DEV uint32_t lanes_below(uint32_t lane) { return (1u << lane) - 1u; }
#ifdef RT_POOL_INLINE_RNG
using PoolRng = PathRng;
#else
using PoolRng = PathRngOol; // one out-of-line Philox for the four phases: the warps of an SM sit in different phases, the instruction caches hold all of them
#endif

template <uint32_t PM, bool WIDE, bool MEDIA, bool GENERAL_MEDIA, bool XF, int P, int MINB>
__global__ void __launch_bounds__(128, MINB) k_pool(const __grid_constant__ DeviceScene S, const __grid_constant__ JobDev J, Queues Q, int64_t* __restrict__ accum) {
    static_assert(P <= 256 && P % 32 == 0, "slot ids are bytes");
    extern __shared__ __align__(16) unsigned char pool_smem[];
    WarpPool<P>& W = reinterpret_cast<WarpPool<P>*>(pool_smem)[threadIdx.x >> 5];
    const unsigned full = 0xffffffffu;
    const uint32_t lane = lane_id(), below = lanes_below(lane);
    const uint32_t DONE = 0xffffffffu;
    const bool planar = (PM & 0x18u) != 0 && (S.flags & 1u) != 0;
    const uint32_t n_inst = XF ? S.n_main_instances : 1u;
    // list lengths (warp-uniform)
    uint32_t n_trace = 0, n_done = 0, n_regen = P, n_mat0 = 0, n_mat1 = 0, n_mat2 = 0, n_mat3 = 0;
    for (uint32_t i = lane; i < (uint32_t)P; i += 32u) W.q_regen[i] = (uint8_t)i;
    __syncwarp();
    unsigned long long chunk_next = 0, chunk_end = 0; // warp-uniform: the warp's chunk of consecutive path indices
    bool exhausted = false;
    // the walk this lane has in flight
    bool have = false;
    uint32_t slot = 0, inst = 0, cur = DONE;
    int sp = 0;
    Ray r; // in the space of instance `inst`
    r.o = mk3(0, 0, 0); r.d = mk3(0, 0, 1); r.time = 0.0;
    RayF f; f.idx = f.idy = f.idz = f.oodx = f.oody = f.oodz = 0.f;
    RayPre pre; pre.a = 1.0; pre.inv_a = 1.0; pre.inv_d = mk3(0, 0, 0);
    BestHit best;
    best_init(best, RT_INF);
    uint32_t stack[WIDE ? 1 : RT_STACK];
    unsigned long long wstack[WIDE ? RT_WIDE_STACK : 1];
    uint32_t my_segments = 0;
    const uint32_t LOW = 16u;    // TRACE ends when no ray waits and at most LOW lanes still walk          (16 / 20 / 24 / 28: 101.2 / 102.1 / 103.0 / 104.0 ms, book-1 final)
    const uint32_t REFILL = 12u; // while rays wait: lanes that must have finished before the warp refills (4 / 8 / 12 / 16: 103.4 / 103.0 / 102.5 / 102.1 ms)

    for (;;) {
        // ================================================================ REGEN
        while (n_regen && !exhausted) {
            const uint32_t take = n_regen < 32u ? n_regen : 32u, base = n_regen - take;
            const unsigned long long avail = chunk_end - chunk_next;
            unsigned long long second_base = 0;
            if (avail < take) {
                if (lane == 0) second_base = atomicAdd(Q.next_path, (unsigned long long)J.chunk);
                second_base = __shfl_sync(full, second_base, 0);
            }
            bool ok = false;
            uint32_t sl = 0;
            if (lane < take) {
                const unsigned long long L = (lane < avail) ? chunk_next + lane : second_base + (lane - avail);
                if (L < J.total_paths) {
                    ok = true;
                    sl = W.q_regen[base + lane];
                    uint32_t s_local, pixel, draw0;
                    split_path_index(L + J.path_base, J.npix_rendered, s_local, pixel);
                    pixel = shard_pixel(J, pixel);
                    const int32_t j = (int32_t)(pixel / (uint32_t)J.W), ii = (int32_t)(pixel - (uint32_t)j * (uint32_t)J.W);
                    const uint64_t path_id = (uint64_t)pixel * (uint64_t)J.spp_total + (uint64_t)(J.sample_begin + (int32_t)s_local);
                    const Ray cr = camera_first_ray<PoolRng>(S.cam, ii, j, J.W, J.H, J.seed, path_id, draw0); // world.rs:1212-1214
                    W.ox[sl] = cr.o.x; W.oy[sl] = cr.o.y; W.oz[sl] = cr.o.z; W.dx[sl] = cr.d.x; W.dy[sl] = cr.d.y; W.dz[sl] = cr.d.z; W.time[sl] = cr.time;
                    W.tr[sl] = 1.f; W.tg[sl] = 1.f; W.tb[sl] = 1.f;
                    W.pixel[sl] = pixel; W.s_local[sl] = s_local; W.draw[sl] = draw0; W.segment[sl] = 0;
                }
            }
            if (avail < take) { chunk_next = second_base + (take - avail); chunk_end = second_base + J.chunk; }
            else chunk_next += take;
            const unsigned okm = __ballot_sync(full, ok);
            if (ok) W.q_trace[n_trace + __popc(okm & below)] = (uint8_t)sl;
            n_trace += __popc(okm);
            if ((uint32_t)__popc(okm) < take) exhausted = true; // path indices past the end: the pool drains from here on
            n_regen = base;
            __syncwarp();
        }
        if (exhausted) n_regen = 0; // slots without a path stay empty

        // ================================================================ TRACE
        for (;;) {
            if (__ballot_sync(full, cur == DONE)) { // a lane finished its walk, or idles
                bool setup = false, commit = false;
                if (have && cur == DONE) {
                    ++inst;
                    if (XF && inst < n_inst) setup = true; // next instance of the main world (hit.rs:660-690: the list scan goes on with closest_so_far)
                    else commit = true;
                }
                const unsigned cm = __ballot_sync(full, commit);
                if (commit) { // world.hit of this slot is complete
                    W.best_t[slot] = best.t;
                    W.best_ref[slot] = best.type == RT_NONE ? RT_POOL_MISS : (best.type << 29) | (best.side << RT_POOL_IDX_BITS) | best.idx;
                    W.best_inst[slot] = (uint8_t)best.inst;
                    W.q_done[n_done + __popc(cm & below)] = (uint8_t)slot;
                    have = false;
                    ++my_segments;
                }
                n_done += __popc(cm);
                const unsigned want = __ballot_sync(full, !have);
                const uint32_t nw = __popc(want), got = nw < n_trace ? nw : n_trace;
                if (!have) {
                    const uint32_t rank = __popc(want & below);
                    if (rank < got) {
                        slot = W.q_trace[n_trace - 1u - rank];
                        have = true; setup = true;
                        inst = 0;
                        best_init(best, RT_INF);
                    }
                }
                n_trace -= got;
                if (setup) {
                    r.o = mk3(W.ox[slot], W.oy[slot], W.oz[slot]);
                    r.d = mk3(W.dx[slot], W.dy[slot], W.dz[slot]);
                    r.time = W.time[slot];
                    uint32_t root;
                    if (XF) {
                        const Instance* ip = &S.instances[inst];
                        xform_ray(S.ops, __ldg(&ip->chain_off), __ldg(&ip->chain_len), r);
                        root = WIDE ? __ldg(&ip->root4) : __ldg(&ip->root);
                    } else {
                        root = WIDE ? S.root4 : __ldg(&S.instances[0].root);
                    }
                    f = make_rayf(r);
                    pre = make_raypre(r, planar);
                    cur = root;
                    sp = 0;
                }
                __syncwarp();
            }
            const uint32_t busy = __popc(__ballot_sync(full, have));
            if (busy == 0) break;
            if (n_trace == 0 && busy <= LOW && n_done != 0) break; // starving: shade what is finished; the walks in flight resume afterwards
            const uint32_t wt = n_trace ? REFILL : ((n_done != 0 && busy > LOW) ? busy - LOW : 1u);
            if (WIDE) walk_wide<PM, true>(S, r, f, pre, 0.001, best, cur, sp, wstack, wt, XF ? inst : 0u);
            else walk_pairs<PM>(S, r, f, pre, 0.001, best, cur, sp, stack, wt, XF ? inst : 0u);
        }
        if (n_done == 0 && !__any_sync(full, have)) break; // every path of this warp has ended and no index is left

        // ================================================================ SHADE 1: classify (and sample the media)
        for (uint32_t base = 0; base < n_done; base += 32u) {
            const uint32_t i = base + lane;
            uint32_t cls = 7u, sl = 0; // 0 Lambertian, 1 Metal / Dielectric, 2 Isotropic, 3 DiffuseLight, 5 ended
            if (i < n_done) {
                sl = W.q_done[i];
                uint32_t ref = W.best_ref[sl];
                if (MEDIA) { // ConstantMedium::hit against closest_so_far (hit.rs:955-986); order independent: keyed draws
                    Ray wr;
                    wr.o = mk3(W.ox[sl], W.oy[sl], W.oz[sl]); wr.d = mk3(W.dx[sl], W.dy[sl], W.dz[sl]); wr.time = W.time[sl];
                    const uint64_t path_id = (uint64_t)W.pixel[sl] * (uint64_t)J.spp_total + (uint64_t)(J.sample_begin + (int32_t)W.s_local[sl]);
                    double closest = W.best_t[sl];
                    int32_t mwin = -1;
                    D3 mp = mk3(0, 0, 0);
                    for (uint32_t mi = 0; mi < S.n_media; ++mi) medium_query<false, GENERAL_MEDIA>(S, mi, wr, 0.001, closest, mwin, mp, J.seed, path_id, (uint32_t)W.segment[sl], nullptr);
                    if (mwin >= 0) {
                        ref = ((uint32_t)PRIM_MEDIUM << 29) | (uint32_t)mwin;
                        W.best_t[sl] = closest;
                        W.best_ref[sl] = ref;
                    }
                }
                if (ref == RT_POOL_MISS) { // world.rs:86-89
                    const F3 bg = miss_color(S, mk3(W.dx[sl], W.dy[sl], W.dz[sl]));
                    accumulate(accum, W.pixel[sl], W.tr[sl] * bg.x, W.tg[sl] * bg.y, W.tb[sl] * bg.z);
                    cls = 5u;
                } else {
                    const uint32_t type = ref >> 29, idx = ref & ((1u << RT_POOL_IDX_BITS) - 1u);
                    const uint32_t mat = (MEDIA && type == PRIM_MEDIUM) ? S.media[idx].mat_id : __ldg(&S.meta[type][idx].mat_id);
                    const uint32_t mt = __ldg(&S.materials[mat].type);
                    cls = mt == MAT_LAMBERTIAN ? 0u : (mt == MAT_ISOTROPIC ? 2u : (mt == MAT_LIGHT ? 3u : 1u));
                }
            }
            unsigned m;
            m = __ballot_sync(full, cls == 0u); if (cls == 0u) W.q_mat[0][n_mat0 + __popc(m & below)] = (uint8_t)sl; n_mat0 += __popc(m);
            m = __ballot_sync(full, cls == 1u); if (cls == 1u) W.q_mat[1][n_mat1 + __popc(m & below)] = (uint8_t)sl; n_mat1 += __popc(m);
            m = __ballot_sync(full, cls == 2u); if (cls == 2u) W.q_mat[2][n_mat2 + __popc(m & below)] = (uint8_t)sl; n_mat2 += __popc(m);
            m = __ballot_sync(full, cls == 3u); if (cls == 3u) W.q_mat[3][n_mat3 + __popc(m & below)] = (uint8_t)sl; n_mat3 += __popc(m);
            m = __ballot_sync(full, cls == 5u); if (cls == 5u) W.q_regen[n_regen + __popc(m & below)] = (uint8_t)sl; n_regen += __popc(m);
        }
        n_done = 0;
        __syncwarp();

        // ================================================================ SHADE 2: per material class, batches of 32
#pragma unroll 1
        for (int c = 0; c < 4; ++c) {
            const uint32_t n_c = c == 0 ? n_mat0 : (c == 1 ? n_mat1 : (c == 2 ? n_mat2 : n_mat3));
            for (uint32_t base = 0; base < n_c; base += 32u) {
                const uint32_t i = base + lane;
                bool cont = false, ended = false;
                uint32_t sl = 0;
                if (i < n_c) {
                    sl = W.q_mat[c][i];
                    Ray wr;
                    wr.o = mk3(W.ox[sl], W.oy[sl], W.oz[sl]); wr.d = mk3(W.dx[sl], W.dy[sl], W.dz[sl]); wr.time = W.time[sl];
                    const uint32_t ref = W.best_ref[sl];
                    HitRec h;
                    if (MEDIA && (ref >> 29) == PRIM_MEDIUM) { // hit.rs:975-984
                        const Medium md = S.media[ref & ((1u << RT_POOL_IDX_BITS) - 1u)];
                        h.t = W.best_t[sl];
                        h.p = medium_point(S, md, wr, h.t);
                        h.n = mk3(0, 0, 0); h.u = 0.0; h.v = 0.0; h.front = true;
                        h.mat = md.mat_id; h.prim_id = md.prim_id;
                    } else {
                        BestHit b;
                        b.t = W.best_t[sl]; b.type = ref >> 29; b.side = (ref >> RT_POOL_IDX_BITS) & 7u; b.idx = ref & ((1u << RT_POOL_IDX_BITS) - 1u);
                        b.inst = W.best_inst[sl];
                        h = finalize_hit<2, PM, XF>(S, wr, b);
                    }
                    const DMaterial m = S.materials[h.mat];
                    const float tr = W.tr[sl], tg = W.tg[sl], tb = W.tb[sl];
                    if (c == 3) { // DiffuseLight: emitted, no scatter (hit.rs:1146-1151, world.rs:78-84)
                        const F3 e = tex_value(S, m.tex, h.u, h.v, h.p);
                        accumulate(accum, W.pixel[sl], tr * e.x, tg * e.y, tb * e.z);
                        ended = true;
                    } else {
                        const uint64_t path_id = (uint64_t)W.pixel[sl] * (uint64_t)J.spp_total + (uint64_t)(J.sample_begin + (int32_t)W.s_local[sl]);
                        PoolRng g;
                        g.init(J.seed, path_id, W.draw[sl]);
                        D3 dir = mk3(0, 0, 0);
                        F3 att = mkf3(0.f, 0.f, 0.f);
                        bool scattered;
                        if (c == 0) scattered = scatter_lambertian(S, m, h.p, h.n, h.u, h.v, g, dir, att);
                        else if (c == 2) scattered = scatter_isotropic(S, m, h.p, h.u, h.v, g, dir, att);
                        else if (m.type == MAT_METAL) scattered = scatter_metal(m, wr.d, h.n, g, dir, att);
                        else scattered = scatter_dielectric(m, wr.d, h.n, h.front, g, dir, att);
                        const uint32_t seg = (uint32_t)W.segment[sl] + 1u;
                        if (scattered && (int32_t)seg < J.max_depth) { // world.rs:64-67, 75
                            W.tr[sl] = tr * att.x; W.tg[sl] = tg * att.y; W.tb[sl] = tb * att.z;
                            W.ox[sl] = h.p.x; W.oy[sl] = h.p.y; W.oz[sl] = h.p.z; W.dx[sl] = dir.x; W.dy[sl] = dir.y; W.dz[sl] = dir.z;
                            W.draw[sl] = g.draw; W.segment[sl] = (uint8_t)seg;
                            cont = true;
                        } else {
                            ended = true; // absorbed (Metal) or depth exhausted: nothing to add
                        }
                    }
                }
                unsigned m2 = __ballot_sync(full, cont);
                if (cont) W.q_trace[n_trace + __popc(m2 & below)] = (uint8_t)sl;
                n_trace += __popc(m2);
                m2 = __ballot_sync(full, ended);
                if (ended) W.q_regen[n_regen + __popc(m2 & below)] = (uint8_t)sl;
                n_regen += __popc(m2);
            }
        }
        n_mat0 = n_mat1 = n_mat2 = n_mat3 = 0;
        __syncwarp();
    }
    uint32_t segs = my_segments;
    for (int o = 16; o > 0; o >>= 1) segs += __shfl_xor_sync(full, segs, o);
    if (lane == 0 && segs) atomicAdd(&Q.stats[0], (unsigned long long)segs);
}

__global__ void k_mega_init(Queues Q) {
    if (threadIdx.x == 0) { *Q.next_path = 0ull; *Q.dead = 0; }
    if (threadIdx.x < 9) Q.stats[threadIdx.x] = 0ull;
}

// ------------------------------------------------------------------ resolve (vec3.rs:89-107 + Screen layout)
__global__ void k_resolve(const int64_t* __restrict__ accum, double* __restrict__ screen, int32_t W, int32_t H, int32_t spp, int32_t rows) {
    const int64_t n = (int64_t)W * H * 3;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t pix = i / 3;
        const int32_t j = (int32_t)(pix / W);
        double out = 0.0;
        if (j < rows) {
            const double sum = (double)accum[i] * (1.0 / 4294967296.0);
            const double scale = 1.0 / (double)spp;
            double c = sqrt(sum * scale);
            c = c < 0.0 ? 0.0 : (c > 1.0 ? 1.0 : c);     // mutil.rs:1-9 (NaN passes through)
            const double q = 255.9 * c;
            out = (q != q) ? 0.0 : (double)(int32_t)q;    // `as i32`: truncation, NaN -> 0
        }
        screen[i] = out;
    }
}

// ------------------------------------------------------------------ reduce + resolve over peer memory (multi-GPU inside the library)
// The one exchange of a sharded render (SURVEY.md 8e) fused with get_normalized_color: this kernel runs on the gathering GPU and reads
// every shard's int64 accumulator where it lies - its own HBM or a peer's, through NVLink / NVSwitch P2P-mapped pointers - adds them
// (integer: order independent, so the image is bit-identical for any shard count) and writes the quantised Screen.  There is no staging
// copy and no separate reduce pass: 24 B per pixel per shard cross the links once, 128 bits per load.
//   sum_out    nullable: the reduced int64 accumulator (rt_render's out_accum)
//   screen_u8  nullable: Screen as bytes, same layout as the f64 Screen (row 0 = bottom, rgb); every value is an integer in 0..255
//   screen_f64 nullable: Screen as the reference's f64 Colors (vec3.rs:89-107)
__global__ void __launch_bounds__(256) k_reduce_resolve(const AccumShards A, int64_t* sum_out /* may alias A.p[0] */, uint8_t* __restrict__ screen_u8,
                                                        double* __restrict__ screen_f64, int32_t W, int32_t H, int32_t spp, int32_t rows) {
    const int64_t n = (int64_t)W * H * 3, n2 = n >> 1; // pairs of channels: 16-byte loads
    const int64_t rendered = (int64_t)W * rows * 3;
    const double scale = 1.0 / (double)spp;
    if (A.need) { // shards rendered by other processes: wait until every peer's stream has published this step (flag in the peer's memory)
        if (threadIdx.x == 0) { // one poller per CTA, the peers one after the other: the flags live in the peers' memory (NVLink reads)
            const long long t0 = clock64();
            for (int g = 0; g < A.n; ++g) {
                const volatile uint32_t* fl = A.ready[g];
                if (!fl) continue;
                while ((int32_t)(*fl - A.need) < 0) {
                    if (clock64() - t0 > 4000000000ll) { // ~2 s at 1.9 GHz: a dead peer must not hang this GPU; the host sees the flag (rt_peer_timed_out)
                        if (A.timeout_flag) *A.timeout_flag = 1u;
                        break;
                    }
                    __nanosleep(500);
                }
            }
        }
        __syncthreads();
        __threadfence_system();
    }
    for (int64_t i2 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i2 < n2 + (n & 1); i2 += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = 2 * i2;
        const bool pair = i + 1 < n;
        long long s0 = 0, s1 = 0;
        for (int g = 0; g < A.n; ++g) {
            if (pair) { // ld.cv: peers rewrite these lines every step; never served from a stale L1 line
                const longlong2 v = __ldcv(reinterpret_cast<const longlong2*>(A.p[g] + i));
                s0 += v.x; s1 += v.y;
            } else {
                s0 += __ldcv(reinterpret_cast<const long long*>(A.p[g] + i));
            }
        }
        if (sum_out) {
            if (pair) *reinterpret_cast<longlong2*>(sum_out + i) = make_longlong2(s0, s1);
            else sum_out[i] = s0;
        }
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            if (k == 1 && !pair) break;
            const int64_t e = i + k;
            double out = 0.0;
            if (e < rendered) { // rows >= `rows` stay (0,0,0): world.rs:1198-1202
                const double sum = (double)(k ? s1 : s0) * (1.0 / 4294967296.0);
                double c = sqrt(sum * scale);
                c = c < 0.0 ? 0.0 : (c > 1.0 ? 1.0 : c);     // mutil.rs:1-9 (NaN passes through)
                const double q = 255.9 * c;
                out = (q != q) ? 0.0 : (double)(int32_t)q;    // `as i32`: truncation, NaN -> 0
            }
            if (screen_u8) screen_u8[e] = (uint8_t)out;
            if (screen_f64) screen_f64[e] = out;
        }
    }
}

// ------------------------------------------------------------------ trace_batch (parity hook)
// WIDE = true: the main world through its 4-wide collapse (scenes that carry one, t_min >= 0), so the parity hook checks the walk the
// render kernels of such a scene use
template <bool WIDE>
__global__ void __launch_bounds__(128) k_trace_batch(const __grid_constant__ DeviceScene S, const rt_ray* __restrict__ rays, int64_t n, double t_min,
                                                     double t_max, int32_t flags, uint64_t seed, rt_hit* __restrict__ out) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        Ray r;
        r.o = mk3(rays[i].o[0], rays[i].o[1], rays[i].o[2]);
        r.d = mk3(rays[i].d[0], rays[i].d[1], rays[i].d[2]);
        r.time = rays[i].time;
        HitRec h;
        const bool hit = world_hit<false, 1, true, true, RT_PM_ALL, true, WIDE>(S, r, t_min, t_max, (flags & RT_TRACE_SEEDED_MEDIA) != 0, seed, (uint64_t)i, 0u, h, nullptr);
        rt_hit o;
        if (hit) {
            o.prim_id = (int32_t)h.prim_id; o.mat_id = (int32_t)h.mat; o.t = h.t;
            o.p[0] = h.p.x; o.p[1] = h.p.y; o.p[2] = h.p.z;
            o.normal[0] = h.n.x; o.normal[1] = h.n.y; o.normal[2] = h.n.z;
            o.u = h.u; o.v = h.v; o.front_face = h.front ? 1 : 0; o.pad_ = 0;
        } else {
            o.prim_id = -1; o.mat_id = -1; o.t = 0.0;
            o.p[0] = o.p[1] = o.p[2] = 0.0; o.normal[0] = o.normal[1] = o.normal[2] = 0.0;
            o.u = o.v = 0.0; o.front_face = 0; o.pad_ = 0;
        }
        out[i] = o;
    }
}

// ------------------------------------------------------------------ unit-level device checks
__global__ void k_unit_op(const __grid_constant__ DeviceScene S, int op, uint32_t ia, uint32_t ib, uint32_t ic, uint32_t id, const double* in, double* out) {
    if (threadIdx.x || blockIdx.x) return;
    if (op == 0) {
        const F3 c = tex_value(S, ia, in[0], in[1], mk3(in[2], in[3], in[4]));
        out[0] = c.x; out[1] = c.y; out[2] = c.z;
    } else if (op == 1) {
        out[0] = perlin_noise(&S.perlin[ia], mk3(in[0], in[1], in[2]));
        out[1] = perlin_turbulence(&S.perlin[ia], mk3(in[0], in[1], in[2]), 7);
    } else if (op == 2) {
        const uint4 r = philox4x32_10(make_uint4(ia, ib, ic, id), make_uint2((uint32_t)in[0], (uint32_t)in[1]));
        out[0] = r.x; out[1] = r.y; out[2] = r.z; out[3] = r.w;
    } else if (op == 3) {
        PathRng g;
        g.init((uint64_t)ia | ((uint64_t)ib << 32), (uint64_t)ic | ((uint64_t)id << 32), 0);
        const double u = (in[0] + g.gen()) / (in[2] - 1.0);
        const double v = (in[1] + g.gen()) / (in[3] - 1.0);
        const Ray r = camera_get_ray(S.cam, u, v, g);
        out[0] = r.o.x; out[1] = r.o.y; out[2] = r.o.z; out[3] = r.d.x; out[4] = r.d.y; out[5] = r.d.z; out[6] = r.time;
    }
}

// ------------------------------------------------------------------ host side
#define CK(x)                                   \
    do {                                        \
        cudaError_t e_ = (x);                   \
        if (e_ != cudaSuccess) { err = e_; goto done; } \
    } while (0)

cudaError_t launch_resolve(const int64_t* d_accum, double* d_screen, int32_t W, int32_t H, int32_t spp, int32_t rows, cudaStream_t stream) {
    const int64_t n = (int64_t)W * H * 3;
    const int blocks = (int)std::min<int64_t>((n + 255) / 256, 148 * 16);
    k_resolve<<<blocks, 256, 0, stream>>>(d_accum, d_screen, W, H, spp, rows);
    return cudaGetLastError();
}

__global__ void k_flag_publish(uint32_t* flag, uint32_t value) {
    __threadfence_system(); // everything this stream wrote before (the render's pixel sums) is visible to peers before the flag is
    *reinterpret_cast<volatile uint32_t*>(flag) = value;
    __threadfence_system();
}
__global__ void k_flag_wait(const uint32_t* flag, uint32_t need, uint32_t* timeout_flag) {
    const volatile uint32_t* fl = flag;
    const long long t0 = clock64();
    while ((int32_t)(*fl - need) < 0) {
        if (clock64() - t0 > 4000000000ll) { *timeout_flag = 1u; break; }
        __nanosleep(200);
    }
    __threadfence_system();
}
cudaError_t launch_flag_publish(uint32_t* flag, uint32_t value, cudaStream_t stream) {
    k_flag_publish<<<1, 1, 0, stream>>>(flag, value);
    return cudaGetLastError();
}
cudaError_t launch_flag_wait(const uint32_t* flag, uint32_t need, uint32_t* timeout_flag, cudaStream_t stream) {
    k_flag_wait<<<1, 1, 0, stream>>>(flag, need, timeout_flag);
    return cudaGetLastError();
}

cudaError_t launch_reduce_resolve(const AccumShards& shards, int64_t* d_sum_out, uint8_t* d_screen_u8, double* d_screen_f64, int32_t W, int32_t H, int32_t spp,
                                  int32_t rows, cudaStream_t stream) {
    const int64_t n2 = ((int64_t)W * H * 3 + 1) / 2;
    const int blocks = (int)std::min<int64_t>((n2 + 255) / 256, 148 * 8);
    k_reduce_resolve<<<blocks, 256, 0, stream>>>(shards, d_sum_out, d_screen_u8, d_screen_f64, W, H, spp, rows);
    return cudaGetLastError();
}

cudaError_t launch_trace_batch(const DeviceScene& scene, const rt_ray* d_rays, int64_t n, double t_min, double t_max, int32_t flags, uint64_t seed,
                               rt_hit* d_out, cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    const int blocks = (int)std::min<int64_t>((n + 127) / 128, 148 * 32);
    if (scene.nodes4 != nullptr && t_min >= 0.0) k_trace_batch<true><<<blocks, 128, 0, stream>>>(scene, d_rays, n, t_min, t_max, flags, seed, d_out);
    else k_trace_batch<false><<<blocks, 128, 0, stream>>>(scene, d_rays, n, t_min, t_max, flags, seed, d_out);
    return cudaGetLastError();
}

cudaError_t launch_unit_op(const DeviceScene& scene, int op, uint32_t ia, uint32_t ib, uint32_t ic, uint32_t id, const double* in8, double* out8) {
    double *d_in = nullptr, *d_out = nullptr;
    cudaError_t err = cudaSuccess;
    CK(cudaMalloc(&d_in, 8 * sizeof(double)));
    CK(cudaMalloc(&d_out, 8 * sizeof(double)));
    CK(cudaMemcpy(d_in, in8, 8 * sizeof(double), cudaMemcpyHostToDevice));
    CK(cudaMemset(d_out, 0, 8 * sizeof(double)));
    k_unit_op<<<1, 32>>>(scene, op, ia, ib, ic, id, d_in, d_out);
    CK(cudaGetLastError());
    CK(cudaMemcpy(out8, d_out, 8 * sizeof(double), cudaMemcpyDeviceToHost));
done:
    cudaFree(d_in);
    cudaFree(d_out);
    return err;
}

struct Workspace { // path state + queues, cached per scene between renders
    char* base = nullptr;
    size_t cap = 0, used = 0;
    uint32_t n_slots = 0;
    PathState P;
    Queues Q;
    unsigned int* h_flag = nullptr;
    cudaEvent_t ev_begin = nullptr, ev_end = nullptr, ev_poll[2] = {nullptr, nullptr};
    template <class T> T* take(size_t n) {
        used = (used + 255) & ~(size_t)255;
        T* p = reinterpret_cast<T*>(base + used);
        used += n * sizeof(T);
        return p;
    }
};

void free_workspace(Workspace* w) {
    if (!w) return;
    if (w->base) cudaFree(w->base);
    if (w->h_flag) cudaFreeHost(w->h_flag);
    if (w->ev_begin) cudaEventDestroy(w->ev_begin);
    if (w->ev_end) cudaEventDestroy(w->ev_end);
    if (w->ev_poll[0]) cudaEventDestroy(w->ev_poll[0]);
    if (w->ev_poll[1]) cudaEventDestroy(w->ev_poll[1]);
    delete w;
}

static cudaError_t ensure_workspace(Workspace*& w, uint32_t N) {
    if (w && w->n_slots == N) return cudaSuccess;
    free_workspace(w);
    w = new Workspace();
    cudaError_t err = cudaSuccess;
    const size_t per_slot = 4 * 32 + 1 + Q_COUNT * 4;
    w->cap = (size_t)N * per_slot + 64 * 256 + 4096;
    if ((err = cudaMalloc(&w->base, w->cap)) != cudaSuccess) return err;
    PathState& P = w->P;
    Queues& Q = w->Q;
    P.A = w->take<SlotA>(N); P.B = w->take<SlotB>(N); P.C = w->take<SlotC>(N); P.D = w->take<SlotD>(N);
    P.alive = w->take<uint8_t>(N);
    for (int q = 0; q < Q_COUNT; ++q) Q.q[q] = w->take<uint32_t>(N);
    Q.counts = w->take<uint32_t>(16);
    Q.dead = w->take<uint32_t>(1);
    Q.ext_cursor = w->take<uint32_t>(1);
    Q.next_path = w->take<unsigned long long>(1);
    Q.stats = w->take<unsigned long long>(9);
    if (w->used > w->cap) return cudaErrorMemoryAllocation;
    if ((err = cudaMallocHost(&w->h_flag, 2 * sizeof(unsigned int))) != cudaSuccess) return err;
    if ((err = cudaEventCreate(&w->ev_begin)) != cudaSuccess) return err;
    if ((err = cudaEventCreate(&w->ev_end)) != cudaSuccess) return err;
    if ((err = cudaEventCreateWithFlags(&w->ev_poll[0], cudaEventDisableTiming)) != cudaSuccess) return err;
    if ((err = cudaEventCreateWithFlags(&w->ev_poll[1], cudaEventDisableTiming)) != cudaSuccess) return err;
    w->n_slots = N;
    return cudaSuccess;
}

template <bool COUNT>
static void launch_extend_p(cudaStream_t st, const DeviceScene& scene, const JobDev& J, const PathState& P, const Queues& Q, int parity) {
    // persistent: exactly the resident number of CTAs (148 SMs x 4); chosen only for media-free scenes with large meshes
    k_extend_p<false, COUNT, 4><<<148 * 4, 128, 0, st>>>(scene, J, P, Q, parity);
}

template <bool MEDIA, bool COUNT>
static void launch_extend(int blocks, bool specialise, bool wide, cudaStream_t st, const DeviceScene& scene, const JobDev& J, const PathState& P, const Queues& Q, int parity) {
    // MINB = resident 128-thread blocks per SM the kernel is compiled for: 4 (128 registers) with generic media code or event
    // counters, 5 (96 registers) otherwise - also for the two primitive-mask-specialised media kernels, which then spill 56-80
    // bytes but gain 5 % (tools/explore.py ab, Cornell smoke 634 -> 668, book-2 final 325 -> 340 Mpaths/s); 6 CTAs/SM (80
    // registers, 130-340 B spilled) is +1 % on Cornell smoke and -1.4 % on book-2 final.  Media whose boundary is one sphere / one box (scene.flags bit 1) use the kernel without
    // the general two-traversal path; the two media scenes of the reference also get their primitive mask compiled in.
    // wide: the counting pass of a scene whose fused kernel walks the 4-wide collapse, and the two specialised media kernels (with
    // the min / max node test they measured 718.7 vs 719.2 (Cornell smoke) and 341.3 vs 341.9 Mpaths/s (book-2 final) against the
    // sibling pairs; with the signed-row test 722 vs 705 and 350 vs 340: profiles/r2_59_ab_ext_wide.txt)
    if constexpr (MEDIA) {
        if (!(scene.flags & 2u)) {
            k_extend<true, COUNT, 4, true><<<blocks, 128, 0, st>>>(scene, J, P, Q, parity);
        } else if (!COUNT && specialise && wide && (scene.prim_mask & ~0x18u) == 0) {
            k_extend<true, false, 5, false, 0x18u, true><<<blocks, 128, 0, st>>>(scene, J, P, Q, parity); // ... on the 4-wide tree
        } else if (!COUNT && specialise && wide && (scene.prim_mask & ~0x1bu) == 0) {
            k_extend<true, false, 5, false, 0x1bu, true><<<blocks, 128, 0, st>>>(scene, J, P, Q, parity);
        } else if (!COUNT && specialise && (scene.prim_mask & ~0x18u) == 0) {
            k_extend<true, false, 5, false, 0x18u><<<blocks, 128, 0, st>>>(scene, J, P, Q, parity); // rects + boxes (Cornell scenes)
        } else if (!COUNT && specialise && (scene.prim_mask & ~0x1bu) == 0) {
            k_extend<true, false, 5, false, 0x1bu><<<blocks, 128, 0, st>>>(scene, J, P, Q, parity); // spheres, moving spheres, rects, boxes (book-2 final)
        } else {
            k_extend<true, COUNT, 4, false><<<blocks, 128, 0, st>>>(scene, J, P, Q, parity);
        }
    } else if constexpr (COUNT) {
        if (wide) k_extend<false, true, 4, false, RT_PM_ALL, true><<<blocks, 128, 0, st>>>(scene, J, P, Q, parity); // counts 4 boxes per wide node visited
        else k_extend<false, true, 4, false><<<blocks, 128, 0, st>>>(scene, J, P, Q, parity);
    } else {
        k_extend<false, false, 5, false><<<blocks, 128, 0, st>>>(scene, J, P, Q, parity);
    }
}

template <uint32_t PM, bool WIDE, bool MEDIA, bool GM, bool XF, int P, int MINB>
static void launch_pool(cudaStream_t st, const DeviceScene& scene, const JobDev& J, const Queues& Q, int64_t* d_accum) {
    auto kern = k_pool<PM, WIDE, MEDIA, GM, XF, P, MINB>;
    const size_t smem = 4 * sizeof(WarpPool<P>); // four warps per CTA, one pool each
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); // per device: set on every launch (microseconds)
    kern<<<148 * MINB, 128, smem, st>>>(scene, J, Q, d_accum);
}
// Resident CTAs per SM of the 4-wide sphere kernels (spheres, + moving spheres, + gravity spheres; no Noise / Image texture): the kernel is
// compiled for it (__launch_bounds__) and launched with 148 x that many CTAs.  6 needs <= 80 registers, 7 <= 72; see
// build/kernels.ptxas.log and tools/reg_pressure.py for what ptxas made of it.  Measured against 5 (profiles/r3_01_ab_occ_sph.txt):
// book-1 final 68.06 -> 64.56 ms (80 registers, no spills), book-1 as shipped 48.98 -> 47.66 ms (80 registers, 52 B of spill stores:
// hit point and normal around the scatter), bouncing-spheres frame 64.34 -> 59.37 ms (no spills).  At 7 all three spill.
#ifndef RT_MEGA_OCC_SPH
#define RT_MEGA_OCC_SPH 6
#endif
template <uint32_t PM>
static void launch_mega_wide_sph(cudaStream_t st, const DeviceScene& scene, const JobDev& J, const Queues& Q, int64_t* d_accum) {
    constexpr int OCC = RT_MEGA_OCC_SPH;
    if (scene.flags & 24u) k_mega<false, 5, false, PM, false, true, true><<<148 * 5, 128, 0, st>>>(scene, J, Q, d_accum); // Perlin / image textures
    else k_mega<false, OCC, false, PM, false, true, false><<<148 * OCC, 128, 0, st>>>(scene, J, Q, d_accum);
}
cudaError_t launch_render(const DeviceScene& scene, const RenderJob& job, const RenderTuning& tune, int64_t* d_accum, cudaStream_t stream,
                          rt_stats* stats, Workspace** wsp) {
    cudaError_t err = cudaSuccess;
    JobDev J;
    J.W = job.width; J.H = job.height; J.rows = job.rows; J.spp_total = job.spp_total;
    J.sample_begin = job.sample_begin; J.max_depth = job.max_depth;
    J.tile_rank = (uint32_t)job.tile_rank; J.tile_count = (uint32_t)std::max(1, job.tile_count);
    uint32_t local_rows = (uint32_t)job.rows;
    if (J.tile_count > 1u) { // rows of [0, rows) whose band belongs to this shard; only the image's last band can be partial
        local_rows = 0;
        for (uint32_t b = J.tile_rank; b * RT_TILE_ROWS < (uint32_t)job.rows; b += J.tile_count)
            local_rows += std::min<uint32_t>(RT_TILE_ROWS, (uint32_t)job.rows - b * RT_TILE_ROWS);
    }
    J.npix_rendered = (uint32_t)job.width * local_rows;
    J.pix_list = job.d_pixels;
    if (job.d_pixels) { J.npix_rendered = job.n_pixels; J.tile_count = 0; } // the caller never combines a list with tile sharding
    J.total_paths = (unsigned long long)J.npix_rendered * (unsigned long long)(job.sample_end - job.sample_begin);
    J.path_base = 0;
    if (job.path_end > job.path_begin) { // a path-range shard of [sample_begin, sample_end): whole samples plus a partial first / last one
        J.path_base = std::min<unsigned long long>(job.path_begin, J.total_paths);
        J.total_paths = std::min<unsigned long long>(job.path_end, J.total_paths) - J.path_base;
    }
    J.seed = job.seed;
    J.count_events = tune.count_events;
    uint32_t N = tune.wave_slots;
    if ((unsigned long long)N > J.total_paths) N = (uint32_t)std::max<unsigned long long>(J.total_paths, 1ull);
    N = (N + 127u) & ~127u;
    J.n_slots = N;

    std::vector<cudaEvent_t> ext_events;
    unsigned long long h_stats[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    uint64_t iterations = 0, launches = 0;
    float ms_device = 0.f;
    double ms_extend = 0.0;
    Workspace* w = nullptr;

    if (J.total_paths == 0) goto done;
    CK(ensure_workspace(*wsp, N));
    w = *wsp;
    {
        PathState& P = w->P;
        Queues& Q = w->Q;
        const int qblocks = (int)std::min<uint32_t>((N + 255) / 256, 148 * 8);
        const bool media = scene.n_media != 0;
        // resident CTAs per SM of the k_extend variant launch_extend picks (only sizes the grid)
        const bool media_specialised = media && (scene.flags & 2u) && tune.prim_specialise && ((scene.prim_mask & ~0x18u) == 0 || (scene.prim_mask & ~0x1bu) == 0);
        const int ext_occ = ((media && !media_specialised) || tune.count_events) ? 4 : 5;
        // measured (profiles/): the warp-scheduled persistent kernel wins on deep triangle BVHs (+22 % on the 871k mesh),
        // the one-ray-per-thread kernel on small scenes and on scenes with media
        const int ext_kind_auto = tune.extend_kind >= 0 ? tune.extend_kind : ((!media && (scene.flags & 4u)) ? 1 : 0);
        // wavefront kernels walk the 4-wide collapse only when it was forced (unmeasured for them) - and in the counting pass of a
        // scene whose fused kernel walks it, so that the device counters describe the tree the timed kernel walks (4 boxes per visit)
        const bool count_wide = tune.count_events && !media && scene.nodes4 != nullptr && tune.bvh_wide != 0;
        const bool ext_wide = count_wide || (media && scene.nodes4 != nullptr && tune.bvh_wide != 0); // see launch_extend
        const int ext_kind = ext_wide ? 0 : ext_kind_auto; // k_extend_p has no wide form
        const int eblocks = (int)std::min<uint32_t>((N + 127) / 128, 148u * (uint32_t)std::max(4, ext_occ) * (uint32_t)std::max(1, tune.extend_waves));
        CK(cudaEventRecord(w->ev_begin, stream));
        // RT_MODE_AUTO (measured on B200, profiles/README.md): the fused persistent kernel wins where shading is cheap
        // (book-1 scenes +20 %, mesh room +7 %); the wavefront wins with media / Perlin textures (Cornell smoke +8 %, book-2 final +56 %)
        const int mode = tune.mode != RT_MODE_AUTO ? tune.mode : ((scene.n_media == 0 && !(scene.flags & 8u)) ? RT_MODE_FUSED : RT_MODE_WAVEFRONT);
        if (mode == RT_MODE_POOL && job.max_depth <= 255 && scene.n_main_instances <= 255u) {
            k_mega_init<<<1, 32, 0, stream>>>(Q);
            {
                const unsigned long long warps = 148ull * 4ull * 4ull;
                unsigned long long c = J.total_paths / (warps * 64ull);
                c = std::max(32ull, std::min((unsigned long long)RT_MEGA_CHUNK, c)) & ~31ull;
                J.chunk = (uint32_t)c;
            }
            const bool wrapper_free = !(scene.flags & 32u) && scene.n_main_instances == 1;
            const bool wide = wrapper_free && scene.nodes4 != nullptr && tune.bvh_wide != 0;
            const uint32_t pmask = scene.prim_mask;
            // opt-in experiment (RT_RENDER_FORCE_POOL / RTB200_MODE=2), four instantiations: measured slower than RT_MODE_AUTO's kernels on
            // every BASELINE config (profiles/README.md, round 2), kept for the A/B and its ncu evidence
            if (media) launch_pool<RT_PM_ALL, false, true, true, true, 128, 4>(stream, scene, J, Q, d_accum);
            else if (wide && pmask == 0x1u) launch_pool<0x1u, true, false, false, false, 128, 4>(stream, scene, J, Q, d_accum);
            else if (wide && (pmask & ~0x28u) == 0) launch_pool<0x28u, true, false, false, false, 128, 4>(stream, scene, J, Q, d_accum);
            else launch_pool<RT_PM_ALL, false, false, false, true, 128, 4>(stream, scene, J, Q, d_accum);
            CK(cudaGetLastError());
            launches += 2;
            iterations = 1;
            if (tune.no_wait) goto done; // RT_RENDER_NO_WAIT: the caller's stream carries on behind the kernel
            CK(cudaEventRecord(w->ev_end, stream));
            CK(cudaMemcpyAsync(h_stats, Q.stats, 9 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, stream));
            CK(cudaStreamSynchronize(stream));
            CK(cudaEventElapsedTime(&ms_device, w->ev_begin, w->ev_end));
            goto done;
        }
        if (mode == RT_MODE_FUSED || mode == RT_MODE_POOL) {
            k_mega_init<<<1, 32, 0, stream>>>(Q);
            // Variant choice (every step A/B-measured on B200, DESIGN.md section 5): compile-time primitive mask when the scene
            // holds only spheres / spheres + moving spheres / rects + triangles; wrapper-free (XF = false) variants at 5 CTAs/SM
            // (96 registers), the 4-wide sphere kernels at RT_MEGA_OCC_SPH (80 registers) unless the scene has Noise / Image textures,
            // everything else at 4 (128 registers); media: 4, or 3 with the general two-traversal path.
            const uint32_t pm = !tune.prim_specialise ? RT_PM_ALL
                                : (scene.prim_mask == 0x1u ? 0x1u : ((scene.prim_mask & ~0x3u) == 0 ? 0x3u : ((scene.prim_mask & ~0x5u) == 0 ? 0x5u : ((scene.prim_mask & ~0x28u) == 0 ? 0x28u : RT_PM_ALL))));
            // Path indices are claimed per warp in chunks of consecutive indices (neighbouring pixels of one sample).  512 is best for
            // long renders (fewer atomics, coherent refills: book-1 final -1.7 % at 128); short renders need smaller chunks or the
            // last chunks leave most warps idle (871k mesh at 10 spp: 127 -> 141 Mpaths/s at 128, 64 at 4096): aim at >= 64 chunks per warp
            // Round 2 (tools/chunk_probe.py, book-1 final): the sphere scenes want the full 512 down to 31-spp renders (62 spp, one of
            // eight strong-scaling shards: 10.98 ms at 96, 10.87 at 512, 11.35 at 1024), so only deep-mesh renders shrink their chunks
            {
                const unsigned long long warps = 148ull * 7ull * 4ull;
                unsigned long long c = J.total_paths / (warps * ((scene.flags & 4u) ? 64ull : 4ull));
                c = std::max(32ull, std::min((unsigned long long)RT_MEGA_CHUNK, c)) & ~31ull;
                J.chunk = (uint32_t)c;
            }
            const bool wrapper_free = !(scene.flags & 32u) && tune.prim_specialise == 2;
            // resumable traversal: +7 % on the 871k-triangle mesh at 20 lanes (round 1), -4 .. -40 % on the sphere scenes, whose shading share
            // is too large to run it with half-empty warps (tools/explore.py ab RTB200_MEGA_WAIT ...)
            // (re-swept on the final kernel, profiles/r2_68_mesh_wait_sweep.txt: 12 / 16 / 20 / 24 / 28 lanes -> 230 / 231.5 / 227 / 215 / 199 Mpaths/s)
            const int mega_wait = tune.mega_wait >= 0 ? tune.mega_wait : ((scene.flags & 4u) ? 16 : 0);
            J.wait_thresh = (uint32_t)std::max(1, std::min(32, mega_wait));
            if (media) {
                if (!(scene.flags & 2u)) k_mega<true, 3, true><<<148 * 3, 128, 0, stream>>>(scene, J, Q, d_accum);
                else k_mega<true, 4, false><<<148 * 4, 128, 0, stream>>>(scene, J, Q, d_accum);
            } else if (wrapper_free && pm != RT_PM_ALL && mega_wait > 0 && scene.n_main_instances == 1) {
                if (pm == 0x1u) k_mega_r<5, 0x1u><<<148 * 5, 128, 0, stream>>>(scene, J, Q, d_accum);
                else if (pm == 0x3u) k_mega_r<5, 0x3u><<<148 * 5, 128, 0, stream>>>(scene, J, Q, d_accum);
                else if (pm == 0x5u) k_mega<false, 5, false, 0x5u, false><<<148 * 5, 128, 0, stream>>>(scene, J, Q, d_accum);
                // the mesh walk is L2-latency bound (long-scoreboard 3.6 per issue): more resident warps beat fewer spills:
                // 5 CTAs/SM (96 regs, 132 B spilled) 126, 6 (80 regs) 134.5, 7 (72 regs, 652 B spilled) 139.7, 8 (64 regs) 135 Mpaths/s
                else if (scene.nodes4 && tune.bvh_wide != 0) {
                    // 4-wide walk: 871k mesh 149.8 -> 179.5 Mpaths/s at 7 CTAs/SM (6: 175.5, 5: 165.9; profiles/r2_00_ab.log)
                    k_mega_r<7, 0x28u, true><<<148 * 7, 128, 0, stream>>>(scene, J, Q, d_accum);
                } else k_mega_r<7, 0x28u><<<148 * 7, 128, 0, stream>>>(scene, J, Q, d_accum);
            } else if (wrapper_free && scene.nodes4 && tune.bvh_wide != 0 && scene.n_main_instances == 1 && (pm == 0x1u || pm == 0x3u || pm == 0x5u || pm == 0x28u)) {
                if (pm == 0x1u) launch_mega_wide_sph<0x1u>(stream, scene, J, Q, d_accum);
                else if (pm == 0x3u) launch_mega_wide_sph<0x3u>(stream, scene, J, Q, d_accum); // motion form (mnodes4)
                else if (pm == 0x5u) launch_mega_wide_sph<0x5u>(stream, scene, J, Q, d_accum);
                else k_mega<false, 5, false, 0x28u, false, true><<<148 * 5, 128, 0, stream>>>(scene, J, Q, d_accum);
            } else if (wrapper_free && pm != RT_PM_ALL) {
                if (pm == 0x1u) k_mega<false, 5, false, 0x1u, false><<<148 * 5, 128, 0, stream>>>(scene, J, Q, d_accum);       // book-1 final
                else if (pm == 0x3u) k_mega<false, 5, false, 0x3u, false><<<148 * 5, 128, 0, stream>>>(scene, J, Q, d_accum);  // book-1 as shipped
                else if (pm == 0x5u) k_mega<false, 5, false, 0x5u, false><<<148 * 5, 128, 0, stream>>>(scene, J, Q, d_accum);  // bouncing-spheres animation (GravitySphere)
                else k_mega<false, 5, false, 0x28u, false><<<148 * 5, 128, 0, stream>>>(scene, J, Q, d_accum);                 // mesh room
            } else if (pm == 0x1u) {
                k_mega<false, 4, false, 0x1u><<<148 * 4, 128, 0, stream>>>(scene, J, Q, d_accum);
            } else if (pm == 0x3u) {
                k_mega<false, 4, false, 0x3u><<<148 * 4, 128, 0, stream>>>(scene, J, Q, d_accum);
            } else if (pm == 0x28u) {
                k_mega<false, 4, false, 0x28u><<<148 * 4, 128, 0, stream>>>(scene, J, Q, d_accum);
            } else {
                k_mega<false, 4, false><<<148 * 4, 128, 0, stream>>>(scene, J, Q, d_accum);
            }
            CK(cudaGetLastError());
            launches += 2;
            iterations = 1;
            if (tune.no_wait) goto done; // RT_RENDER_NO_WAIT: the caller's stream carries on behind the kernel
            CK(cudaEventRecord(w->ev_end, stream));
            CK(cudaMemcpyAsync(h_stats, Q.stats, 9 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, stream));
            CK(cudaStreamSynchronize(stream));
            CK(cudaEventElapsedTime(&ms_device, w->ev_begin, w->ev_end));
            goto done;
        }
        k_init<<<qblocks, 256, 0, stream>>>(P, Q, N);
        CK(cudaGetLastError());
        ++launches;
        int parity = 0;   // counts buffer the next k_shade_all drains
        const int batch = 16; // iterations enqueued between completion checks
        int pending = -1;
        bool finished = false;
        w->h_flag[0] = w->h_flag[1] = 0;
        for (uint64_t guard = 0; !finished && guard < (1ull << 40); ++guard) {
            const int slot = (int)(guard & 1);
            for (int it = 0; it < batch; ++it) {
                k_shade_all<<<qblocks, 256, 0, stream>>>(scene, J, P, Q, d_accum, parity);
                parity ^= 1;
                cudaEvent_t ea = nullptr, eb = nullptr;
                if (tune.timed_extend) {
                    CK(cudaEventCreate(&ea)); CK(cudaEventCreate(&eb));
                    CK(cudaEventRecord(ea, stream));
                }
                if (ext_kind == 1 && !media) {
                    if (tune.count_events) launch_extend_p<true>(stream, scene, J, P, Q, parity); else launch_extend_p<false>(stream, scene, J, P, Q, parity);
                } else if (media) {
                    if (tune.count_events) launch_extend<true, true>(eblocks, tune.prim_specialise != 0, ext_wide, stream, scene, J, P, Q, parity); else launch_extend<true, false>(eblocks, tune.prim_specialise != 0, ext_wide, stream, scene, J, P, Q, parity);
                } else {
                    if (tune.count_events) launch_extend<false, true>(eblocks, tune.prim_specialise != 0, ext_wide, stream, scene, J, P, Q, parity); else launch_extend<false, false>(eblocks, tune.prim_specialise != 0, ext_wide, stream, scene, J, P, Q, parity);
                }
                if (tune.timed_extend) {
                    CK(cudaEventRecord(eb, stream));
                    ext_events.push_back(ea); ext_events.push_back(eb);
                }
                ++iterations;
                launches += 2;
            }
            CK(cudaGetLastError());
            CK(cudaMemcpyAsync(&w->h_flag[slot], Q.dead, sizeof(unsigned int), cudaMemcpyDeviceToHost, stream));
            CK(cudaEventRecord(w->ev_poll[slot], stream));
            if (pending >= 0) {
                CK(cudaEventSynchronize(w->ev_poll[pending]));
                if (w->h_flag[pending] >= N) finished = true;
            }
            pending = slot;
        }
        CK(cudaEventRecord(w->ev_end, stream));
        CK(cudaMemcpyAsync(h_stats, Q.stats, 9 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
        CK(cudaEventElapsedTime(&ms_device, w->ev_begin, w->ev_end));
        for (size_t i = 0; i + 1 < ext_events.size(); i += 2) {
            float ms = 0.f;
            CK(cudaEventElapsedTime(&ms, ext_events[i], ext_events[i + 1]));
            ms_extend += ms;
        }
    }
done:
    if (stats) {
        stats->paths = J.total_paths;
        stats->segments = h_stats[0];
        stats->box_tests = h_stats[1];
        stats->prim_tests[0] = h_stats[2];
        for (int m = 0; m < 5; ++m) stats->scatters[m] = h_stats[4 + m];
        stats->iterations = iterations;
        stats->kernel_launches = launches;
        stats->ms_device = ms_device;
        stats->ms_extend = ms_extend;
    }
    for (cudaEvent_t e : ext_events) cudaEventDestroy(e);
    return err;
}

} // namespace rtb
