// kernels.h — host-callable launchers of the sm_100a kernels (implemented in kernels.cu).
#pragma once
#include <cuda_runtime.h>

#include <vector>
#include <stdint.h>

#include "../../../include/rtb200.h"
#include "../rt_types.h"

namespace rtb {

struct RenderJob {
    int32_t width, height, rows;      // rows = rendered rows (compat_threads quirk), rows <= height
    int32_t spp_total;                // Config.samples_per_pixel (for path ids and the final divide)
    int32_t sample_begin, sample_end; // this call's shard
    int32_t max_depth;
    uint64_t seed;
    int32_t tile_rank = 0, tile_count = 1; // RT_RENDER_TILE_SHARD: this call renders the row bands b with b % tile_count == tile_rank
    // rt_render_device_paths: only the path indices [path_begin, path_end) of the call's (pixels x samples) in sample-major order
    // (index = sample * pixels + pixel); 0, 0 = all of them
    uint64_t path_begin = 0, path_end = 0;
    // rt_render_adaptive: render only the n_pixels pixels of this device list (ascending global pixel indices) instead of the rows
    // [0, rows); path index = sample * n_pixels + list position.  null = every pixel of [0, rows)
    const uint32_t* d_pixels = nullptr;
    uint32_t n_pixels = 0;
};

#define RT_MODE_WAVEFRONT 0 // k_extend + k_shade_all per iteration, per-material queues, path state in HBM
#define RT_MODE_FUSED 1     // k_mega: persistent threads, path state in registers
#define RT_MODE_POOL 2      // k_pool: warp-local wavefront, path state and per-material slot lists in shared memory
#define RT_MODE_AUTO (-1)    // measured rule: fused for scenes without media and without noise textures, else wavefront

struct RenderTuning {
    int mode = RT_MODE_AUTO;
    int bvh_builder = 0;            // 0 = host binned SAH (best trees), 1 = device LBVH for instances of >= bvh_device_min primitives (fast commit)
    int bvh_device_min = 4096;
    int mega_wait = -1;             // k_mega_r (resumable traversal): finished lanes that end a traversal round; 0 = plain k_mega, -1 = auto (20 on large meshes)
    uint32_t wave_slots = 1u << 20; // resident paths (path-state slots)
    int timed_extend = 0;           // 1: bracket every extend launch with CUDA events (for the roofline)
    int count_events = 0;           // 1: count BVH node visits / primitive tests on the device
    int extend_kind = -1;           // 0: one ray per thread (while-while), 1: persistent warp-scheduled k_extend_p, -1: auto (1 for big meshes without media)
    int prim_specialise = 2;        // 1: kernel variants compiled for the primitive types the scene contains; 2: also without wrapper handling for wrapper-free scenes; 0: generic
    int bvh_wide = -1;              // 4-wide collapse of a single wrapper-free instance's tree for the fused kernels: 1 build it where possible, 0 never, -1 auto (plain-sphere scenes and large meshes; RTB200_BVH_WIDE)
    int no_wait = 0;                // RT_RENDER_NO_WAIT: single-launch modes return after enqueueing
    int extend_waves = 4;           // k_extend grid = 148 SMs * resident CTAs * extend_waves blocks (grid-stride over the slots)
};

// Wavefront render of one shard into a device-resident int64 fixed-point accumulator (W*H*3).
// Returns cudaSuccess or the first CUDA error; fills stats.
struct Workspace; // path state + queues, allocated on first use and reused by later renders of the scene
void free_workspace(Workspace* w);
cudaError_t launch_render(const DeviceScene& scene, const RenderJob& job, const RenderTuning& tune, int64_t* d_accum, cudaStream_t stream,
                          rt_stats* stats, Workspace** workspace);

// accum -> Screen-layout doubles (vec3.rs:89-107), rows >= rendered_rows stay 0
cudaError_t launch_resolve(const int64_t* d_accum, double* d_screen, int32_t width, int32_t height, int32_t spp, int32_t rendered_rows,
                           cudaStream_t stream);

// Sum of the shards' accumulators + resolve in one pass; the pointers may address peer GPUs' memory (P2P over NVLink).
#define RT_MAX_GPUS 16
struct AccumShards {
    const int64_t* p[RT_MAX_GPUS];
    int32_t n;
    // Cross-process shards (rt_peer_*, one process per GPU): shard g is complete once *ready[g] >= need (a flag in the peer's own
    // allocation, written by its stream after its render); the kernel waits for that itself.  need == 0: no waiting (one process).
    const uint32_t* ready[RT_MAX_GPUS];
    uint32_t need;
    uint32_t* timeout_flag; // set to 1 when a wait gave up (nullable)
};
// one-thread flag kernels of the peer group: publish writes `value` to a flag after a system-wide fence; wait spins until a (peer's)
// flag reaches `need` (bounded: ~2 s, then *timeout_flag = 1 and it gives up instead of hanging the GPU)
cudaError_t launch_flag_publish(uint32_t* flag, uint32_t value, cudaStream_t stream);
cudaError_t launch_flag_wait(const uint32_t* flag, uint32_t need, uint32_t* timeout_flag, cudaStream_t stream);
cudaError_t launch_reduce_resolve(const AccumShards& shards, int64_t* d_sum_out, uint8_t* d_screen_u8, double* d_screen_f64, int32_t W, int32_t H, int32_t spp,
                                  int32_t rows, cudaStream_t stream);

// ---- adaptive sampling (adaptive.cu, rt_render_adaptive / rt_render_adaptive_multi)
// The half accumulators A and B of every GPU that renders rounds (n = 1: the scene's own GPU); the kernels read them where they lie,
// like k_reduce_resolve reads AccumShards, and add the int64 components of a pixel before any f64 arithmetic.  Every pointer must be
// 16-byte aligned: the kernels read pixel pairs and channel pairs with 128-bit loads (A and B of one allocation start at even offsets).
struct AdaptiveShards {
    const int64_t* a[RT_MAX_GPUS];
    const int64_t* b[RT_MAX_GPUS];
    int32_t n;
};
// Check point after n samples (n / 2 in each of the half accumulators A and B) over the active list d_list_in: the half-buffer error of
// every active pixel into the byte mask d_u (W * rows), its box dilation restricted to the active set into d_keep, the final count n
// into d_samples for the pixels that leave, and the stable compaction of the pixels that stay into d_list_out; their number is written
// to *count_out (may be pinned host memory).
struct AdaptiveCheck {
    AdaptiveShards shards;
    const uint32_t* d_list_in;
    uint32_t n_active;
    uint32_t* d_list_out;
    uint32_t* count_out;
    uint8_t* d_u;
    uint8_t* d_keep;
    int32_t* d_samples;
    void* d_temp;        // CUB temp storage of adaptive_select_temp_bytes(n_active or more) bytes
    size_t temp_bytes;
    int32_t W, rows, n, radius;
    double threshold;
};
cudaError_t launch_adaptive_iota(uint32_t* d_list, uint32_t n, cudaStream_t stream); // d_list[i] = i
size_t adaptive_select_temp_bytes(uint32_t max_items);
cudaError_t launch_adaptive_check(const AdaptiveCheck& c, cudaStream_t stream);
cudaError_t launch_adaptive_fill(const uint32_t* d_list, uint32_t n_active, int32_t n, int32_t* d_samples, cudaStream_t stream); // samples[list[q]] = n
// accum_out = the sum of every shard's A + B, Screen bytes resolved with each pixel's own sample count (0 samples: black)
cudaError_t launch_resolve_adaptive(const AdaptiveShards& shards, const int32_t* d_samples, int64_t* d_accum_out, uint8_t* d_screen_u8, int32_t W,
                                    int32_t H, cudaStream_t stream);

// world.hit for n rays (device pointers)
cudaError_t launch_trace_batch(const DeviceScene& scene, const rt_ray* d_rays, int64_t n, double t_min, double t_max, int32_t flags, uint64_t seed,
                               rt_hit* d_out, cudaStream_t stream);

// unit-level device checks (E3): evaluates single device functions on small inputs
// op 0: tex_value(tex = ia, u = in[0], v = in[1], p = in[2..5)) -> out[0..3)
// op 1: perlin noise / turbulence of perlin table ia at p = in[0..3) -> out[0], out[1]
// op 2: philox block ctr = (ia, ib, ic, id) key = (in[0], in[1]) as u32 -> out[0..4) as doubles
// op 3: camera ray for (seed = ia|ib<<32, path_id = ic|id<<32, i = in[0], j = in[1], W = in[2], H = in[3]) -> out[0..7)
// Device-side LBVH build of one instance (lbvh.cu, SURVEY.md 8(f) n1); *ok = false -> use the host builder.
cudaError_t lbvh_build_device(const float* h_boxes, const uint8_t* h_types, uint32_t n, uint32_t max_leaf, uint32_t base, uint32_t type_cursor[PRIM_TYPE_COUNT],
                              std::vector<BvhNode32>& out_nodes, std::vector<uint32_t>& leaf_order, int* max_depth, float* ms_device, bool* ok);

cudaError_t launch_unit_op(const DeviceScene& scene, int op, uint32_t ia, uint32_t ib, uint32_t ic, uint32_t id, const double* in8, double* out8);

} // namespace rtb
