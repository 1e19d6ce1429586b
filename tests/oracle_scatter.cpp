// TEST INFRASTRUCTURE ONLY.  One level of the oracle's ray_color (oracle/oracle.cpp) for caller rays, the reference
// for rt_scatter_batch: collection_ray_intersect, then material_scatter / material_emitted or background, with the
// Philox PathRng keyed (seed; keys[2i], keys[2i+1]) at event level + 1.  Built from the oracle's own functions against
// oracle/liboracle.so (tests/scatter_oracle.py); compile with the oracle's flags (-ffp-contract=off -fno-fast-math).
#include <cstring>

#include "../oracle/oracle.hpp"

using namespace orc;

extern "C" void orc_scatter_batch(const void* sv, const rt_ray* rays, const uint32_t* keys, uint64_t n, uint32_t level,
                                  uint64_t seed, double t_min, double t_max, int32_t* shape_index, double* t,
                                  uint8_t* outcome, rt_vec3* color, rt_ray* scattered) {
    const Scene& sc = *(const Scene*)sv;
    PathRng rng;
    rng.mode = RNG_PHILOX;
    rng.key[0] = (uint32_t)seed;
    rng.key[1] = (uint32_t)(seed >> 32);
    for (uint64_t i = 0; i < n; i++) {
        const Ray r{V3{rays[i].origin.x, rays[i].origin.y, rays[i].origin.z},
                    V3{rays[i].direction.x, rays[i].direction.y, rays[i].direction.z}};
        Hit h;
        const bool found = collection_ray_intersect(sc, r, t_min, t_max, &h, nullptr);
        V3 col = v3(0.0, 0.0, 0.0);
        Ray out{v3(0.0, 0.0, 0.0), v3(0.0, 0.0, 0.0)};
        uint8_t oc = RT_BOUNCE_MISS;
        if (!found) {
            col = background(r);
        } else {
            const rt_material& m = sc.materials[sc.shapes[h.shape].material];
            rng.pixel = keys[2 * i];
            rng.sample = keys[2 * i + 1];
            rng.begin_event(level + 1);
            Ray s;
            if (material_scatter(sc, m, r, h, rng, &s, &col)) {
                oc = RT_BOUNCE_SCATTER;
                out = s;
            } else {
                oc = RT_BOUNCE_EMIT;
                col = material_emitted(sc, m, h.u, h.v, h.point);
            }
        }
        if (shape_index) shape_index[i] = found ? h.shape : -1;
        if (t) t[i] = found ? h.distance : 0.0;
        if (outcome) outcome[i] = oc;
        if (color) color[i] = rt_vec3{col.x, col.y, col.z};
        if (scattered)
            scattered[i] = rt_ray{rt_vec3{out.origin.x, out.origin.y, out.origin.z},
                                  rt_vec3{out.direction.x, out.direction.y, out.direction.z}};
    }
}
