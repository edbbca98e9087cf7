/* tests/oracle_occlusion.c — TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * The occlusion queries of tcrt_occluded_rays / tcrt_occluded_lights (include/tcrt.h) restated on the CPU with the pinned
 * oracle's own code: in_shade (inShadeCollisionDetection) applied to caller-supplied rays with their limits, and to
 * (point, light) pairs built as shade_lights builds its shadow rays, with the calls' validity rules and 0xFF markers.  It
 * also exports the shadow-ray origins of a frame's eye rays: h.P of build_hit, which carries the 1e-3 normal offset of
 * planes.  oracle/tcrt_oracle.c is included unchanged.  Built by tests/test_occlusion.py with the oracle's flags:
 *   gcc -std=gnu11 -O2 -fPIC -shared -ffp-contract=off oracle_occlusion.c -lm
 */
#include "../oracle/tcrt_oracle.c"

static int origin_valid(const float* o) {
    for (int k = 0; k < 3; k++)
        if (!isfinite(o[k]) || fabsf(o[k]) > 1099511627776.0f) return 0;   /* 2^40 */
    return 1;
}

/* the ray batches' direction rule: s = (dx*dx + dy*dy) + dz*dz unfused, |s - 1| <= 2^-21 (NaN fails) */
static int direction_valid(v3 d) {
    const float s = (d.x * d.x + d.y * d.y) + d.z * d.z;
    return fabsf(s - 1.0f) <= 4.76837158203125e-07f;
}

/* occluded[i] for rays [0, n): 1, 0, or 0xFF for a ray outside the batch rule or a tmax that is NaN or <= 0.
 * *n_invalid and *n_tests (may be NULL) count the refused and the traced rays.  Returns 0, or -1. */
int tcrt_oracle_occluded_rays(const tcrt_scene* s, size_t n, const float* origins, int shared, const float* dirs,
                              const float* tmax, unsigned char* occluded, unsigned long long* n_invalid,
                              unsigned long long* n_tests) {
    if (!s || (n && (!origins || !dirs || !tmax || !occluded))) return -1;
    oracle_counters c;
    memset(&c, 0, sizeof(c));
    g_cnt = &c;
    unsigned long long bad = 0, traced = 0;
    for (size_t i = 0; i < n; i++) {
        const float* o = origins + (shared ? 0 : 3 * i);
        const v3 D = v3_ld(dirs + 3 * i);
        const int ok = origin_valid(o) && isfinite(D.x) && isfinite(D.y) && isfinite(D.z) && direction_valid(D) &&
                       tmax[i] > 0.0f;
        if (!ok) {
            occluded[i] = 0xFF;
            bad++;
            continue;
        }
        traced++;
        occluded[i] = (unsigned char)in_shade(s, v3_ld(o), D, tmax[i], &c);
    }
    if (n_invalid) *n_invalid = bad;
    if (n_tests) *n_tests = traced;
    return 0;
}

/* occluded[i * n_lights + l] for points [0, n) and every light, built as shade_lights builds its shadow ray (inShade,
 * RayTracer.cpp:743-771): dir = L - P, dist = |dir|, lr = dir / dist.  0xFF for a point outside the origin rule or an lr
 * outside the direction rule.  Counts in pairs.  Returns 0, or -1. */
int tcrt_oracle_occluded_lights(const tcrt_scene* s, size_t n, const float* points, unsigned char* occluded,
                                unsigned long long* n_invalid, unsigned long long* n_tests) {
    if (!s || (n && (!points || !occluded))) return -1;
    oracle_counters c;
    memset(&c, 0, sizeof(c));
    g_cnt = &c;
    unsigned long long bad = 0, traced = 0;
    const size_t nl = (size_t)s->n_lights;
    for (size_t i = 0; i < n; i++) {
        const float* pp = points + 3 * i;
        const int p_ok = origin_valid(pp);
        const v3 P = v3_ld(pp);
        for (size_t l = 0; l < nl; l++) {
            const int lo = s->light_obj[l];
            /* shade_lights, tcrt_oracle.c: the shadow ray of light l from P */
            v3 Lpos = v3_ld(s->obj_origin + 4 * lo);
            v3 dir = v3_sub(Lpos, P);
            float dist = sqrtf(dir.x * dir.x + dir.y * dir.y + dir.z * dir.z);
            v3 lr = v3_make(dir.x / dist, dir.y / dist, dir.z / dist);
            if (!p_ok || !direction_valid(lr)) {
                occluded[i * nl + l] = 0xFF;
                bad++;
                continue;
            }
            traced++;
            occluded[i * nl + l] = (unsigned char)in_shade(s, P, lr, dist, &c);
        }
    }
    if (n_invalid) *n_invalid = bad;
    if (n_tests) *n_tests = traced;
    return 0;
}

/* The shadow-ray origins of the eye rays of columns [x0, x1) (x-major like frames): P[3k..] = h.P of the primary hit, and
 * kind[k] = 1 for a non-light hit (its shadow rays start at P), 2 for a light, 0 for a miss (P = 0 for both).  Returns 0,
 * or -1. */
int tcrt_oracle_shadow_origins(const tcrt_scene* s, const tcrt_camera* cam, const tcrt_params* p, int x0, int x1,
                               float* P, unsigned char* kind) {
    if (!s || !cam || !p || !P || !kind || x0 < 0 || x1 > p->width || x0 > x1) return -1;
    oracle_counters c;
    memset(&c, 0, sizeof(c));
    g_cnt = &c;
    size_t k = 0;
    for (int x = x0; x < x1; x++)
        for (int z = 0; z < p->height; z++, k++) {
            v3 O, D;
            primary_ray(cam, p, x, z, &O, &D);
            float dist, px, py, den;
            const int obj = nearest_hit(s, p, O, D, &dist, &px, &py, &den, &c);
            P[3 * k] = P[3 * k + 1] = P[3 * k + 2] = 0.0f;
            kind[k] = 0;
            if (obj < 0) continue;
            hit_record h;
            build_hit(s, obj, dist, px, py, den, O, D, &h);
            kind[k] = h.is_light ? 2 : 1;
            if (h.is_light) continue;
            P[3 * k] = h.P.x;
            P[3 * k + 1] = h.P.y;
            P[3 * k + 2] = h.P.z;
        }
    return 0;
}
