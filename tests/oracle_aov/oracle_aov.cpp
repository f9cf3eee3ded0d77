// oracle_aov.cpp — TEST INFRASTRUCTURE (tests/test_denoise.py).  The CPU oracle (oracle/oracle_capi.cpp, compiled into this library
// as it is) plus orc_render_aov: the first-hit feature sums of include/rtb200.h's RTB_FN(render_aov), restated in f64 on the oracle's
// own scene, camera, world.hit and material types.  Build flags are oracle/Makefile's.
#include "../../oracle/oracle_capi.cpp"

namespace {
double clamp01(double x) { return x < 0.0 ? 0.0 : (x > 1.0 ? 1.0 : x); }
} // namespace

extern "C" {

int32_t orc_render_aov(rt_scene* s, const rt_render_config* cfg, int64_t* out_albedo, int64_t* out_normal, rt_stats* stats) {
    CHECK_SCENE(s);
    if (!cfg) return fail(RT_ERR_INVALID, "null config");
    if (RT_RENDER_TILE_COUNT(cfg->flags) > 1 || (cfg->flags & RT_RENDER_NO_WAIT)) return fail(RT_ERR_INVALID, "tile shard / no-wait");
    if (!s->committed) return fail(RT_ERR_STATE, "scene not committed");
    if (!s->has_cam) return fail(RT_ERR_STATE, "no camera");
    if (cfg->image_width <= 0 || cfg->samples_per_pixel <= 0 || cfg->max_depth <= 0) return fail(RT_ERR_INVALID, "Config assert");
    const int32_t W = cfg->image_width, H = orc_image_height(cfg);
    if (H <= 0) return fail(RT_ERR_INVALID, "image height <= 0");
    const int32_t spp = cfg->samples_per_pixel, s0 = cfg->sample_begin, s1 = cfg->sample_end == 0 ? spp : cfg->sample_end;
    if (s0 < 0 || s1 > spp || s0 > s1) return fail(RT_ERR_INVALID, "bad sample range");
    const int32_t rows = cfg->compat_threads > 0 ? (H / cfg->compat_threads) * cfg->compat_threads : H;
    const size_t n = (size_t)W * H * 3;
    std::vector<int64_t> alb(n, 0), nor(n, 0);
    const Hittable& world = *s->root;
    auto fix = [](double x) { return (int64_t)std::nearbyint(x * 4294967296.0); }; // round to nearest even (default rounding mode)
    PathCtx c;
    tls_ctx() = &c;
    for (int32_t j = 0; j < rows; ++j)
        for (int32_t i = 0; i < W; ++i)
            for (int32_t sidx = s0; sidx < s1; ++sidx) {
                const uint64_t path_id = ((uint64_t)j * (uint64_t)W + (uint64_t)i) * (uint64_t)spp + (uint64_t)sidx;
                c.begin_path(cfg->seed, path_id); // segment 0: the medium draws of the render's first world.hit
                c.cnt.paths++;
                c.cnt.segments++;
                const double u = ((double)i + c.gen()) / (double)(W - 1);
                const double v = ((double)j + c.gen()) / (double)(H - 1);
                const Ray r = s->cam.get_ray(u, v);
                HitRecord rec;
                Color a(0, 0, 0);
                Vec3 nn(0, 0, 0);
                if (!world.hit(r, 0.001, INF, rec)) {
                    const Color bg = s->background.at(r);
                    a = Color(clamp01(bg.x), clamp01(bg.y), clamp01(bg.z));
                } else {
                    const Material* m = rec.mat_ptr;
                    nn = rec.normal;
                    if (const Lambertian* l = dynamic_cast<const Lambertian*>(m)) a = l->albedo->value(rec.u, rec.v, rec.p);
                    else if (const Metal* me = dynamic_cast<const Metal*>(m)) a = me->albedo;
                    else if (dynamic_cast<const Dielectric*>(m)) a = Color(1, 1, 1);
                    else if (const DiffuseLight* dl = dynamic_cast<const DiffuseLight*>(m)) {
                        const Color e = dl->emitted(rec.u, rec.v, rec.p);
                        a = Color(clamp01(e.x), clamp01(e.y), clamp01(e.z));
                    } else if (const Isotropic* is = dynamic_cast<const Isotropic*>(m)) {
                        a = is->albedo->value(rec.u, rec.v, rec.p);
                        nn = Vec3(0, 0, 0);
                    }
                }
                const size_t e = ((size_t)j * W + i) * 3;
                alb[e] += fix(a.x); alb[e + 1] += fix(a.y); alb[e + 2] += fix(a.z);
                nor[e] += fix(nn.x); nor[e + 1] += fix(nn.y); nor[e + 2] += fix(nn.z);
            }
    tls_ctx() = nullptr;
    if (out_albedo) std::memcpy(out_albedo, alb.data(), n * sizeof(int64_t));
    if (out_normal) std::memcpy(out_normal, nor.data(), n * sizeof(int64_t));
    if (stats) {
        std::memset(stats, 0, sizeof *stats);
        stats->paths = c.cnt.paths;
        stats->segments = c.cnt.segments;
    }
    return RT_OK;
}

} // extern "C"
