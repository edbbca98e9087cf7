/* tests/oracle_rays.c — TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * The ray batches of tcrt_trace_rays / tcrt_intersect_rays (include/tcrt.h) restated on the CPU with the pinned oracle's
 * own code: trace_pixel (calculatePixel at level 0) and nearest_hit + the n2 of build_hit, applied to caller-supplied rays,
 * with the batch's validity rule and invalid markers.  oracle/tcrt_oracle.c is included unchanged.  Built by
 * tests/test_ray_batches.py with the oracle's flags:
 *   gcc -std=gnu11 -O2 -fPIC -shared -ffp-contract=off oracle_rays.c -lm
 */
#include "../oracle/tcrt_oracle.c"

/* The validity rule: all six components finite, |o_k| <= 2^40, s = (dx*dx + dy*dy) + dz*dz (binary32, unfused) with
 * |s - 1| <= 2^-21.  1 valid, 0 not. */
int tcrt_oracle_ray_valid(const float* o, const float* d) {
    for (int k = 0; k < 3; k++)
        if (!isfinite(o[k]) || !isfinite(d[k]) || fabsf(o[k]) > 1099511627776.0f) return 0;
    const float s = (d[0] * d[0] + d[1] * d[1]) + d[2] * d[2];
    return fabsf(s - 1.0f) <= 4.76837158203125e-07f;
}

static const float* ray_origin(const float* origins, int shared, size_t i) { return origins + (shared ? 0 : 3 * i); }

/* Colours of rays [0, n) into rgb[3i..]; counters may be NULL.  *n_invalid gets the refused rays.  Returns 0, or -1. */
int tcrt_oracle_trace_rays(const tcrt_scene* s, const tcrt_params* p, size_t n, const float* origins, int shared,
                           const float* dirs, float* rgb, unsigned long long* n_invalid, oracle_counters* counters) {
    if (!s || !p || (n && (!origins || !dirs || !rgb)) || p->max_depth < 0) return -1;
    oracle_counters c;
    memset(&c, 0, sizeof(c));
    g_cnt = &c;
    level_rec* stack = (level_rec*)malloc(sizeof(level_rec) * (size_t)(p->max_depth + 2));
    if (!stack) return -1;
    unsigned long long bad = 0;
    for (size_t i = 0; i < n; i++) {
        const float* o = ray_origin(origins, shared, i);
        const float* d = dirs + 3 * i;
        if (!tcrt_oracle_ray_valid(o, d)) {
            union { unsigned u; float f; } nan = {0x7fc00000u};
            rgb[3 * i] = rgb[3 * i + 1] = rgb[3 * i + 2] = nan.f;
            bad++;
            continue;
        }
        c.rays_primary++;
        v3 col = trace_pixel(s, p, v3_ld(o), v3_ld(d), stack, &c);
        rgb[3 * i] = col.x;
        rgb[3 * i + 1] = col.y;
        rgb[3 * i + 2] = col.z;
    }
    free(stack);
    if (n_invalid) *n_invalid = bad;
    if (counters) *counters = c;
    return 0;
}

/* Nearest hits of rays [0, n): obj[i], dist[i], normal[3i..3i+2]; a miss is -1, far_dist, (+0, +0, +0), an invalid ray
 * -2, NaN, NaN.  Returns 0, or -1. */
int tcrt_oracle_intersect_rays(const tcrt_scene* s, const tcrt_params* p, size_t n, const float* origins, int shared,
                               const float* dirs, int* obj, float* dist, float* normal, unsigned long long* n_invalid) {
    if (!s || !p || (n && (!origins || !dirs || !obj || !dist || !normal))) return -1;
    oracle_counters c;
    memset(&c, 0, sizeof(c));
    g_cnt = &c;
    unsigned long long bad = 0;
    for (size_t i = 0; i < n; i++) {
        const float* o = ray_origin(origins, shared, i);
        const float* d = dirs + 3 * i;
        if (!tcrt_oracle_ray_valid(o, d)) {
            union { unsigned u; float f; } nan = {0x7fc00000u};
            obj[i] = -2;
            dist[i] = normal[3 * i] = normal[3 * i + 1] = normal[3 * i + 2] = nan.f;
            bad++;
            continue;
        }
        const v3 O = v3_ld(o), D = v3_ld(d);
        float t, px, py, den;
        const int k = nearest_hit(s, p, O, D, &t, &px, &py, &den, &c);
        v3 nn = v3_make(0.0f, 0.0f, 0.0f);
        if (k >= 0) {
            hit_record h;
            build_hit(s, k, t, px, py, den, O, D, &h);
            nn = h.n2;
        }
        obj[i] = k;
        dist[i] = t;   /* nearest_hit leaves far_dist on a miss */
        normal[3 * i] = nn.x;
        normal[3 * i + 1] = nn.y;
        normal[3 * i + 2] = nn.z;
    }
    if (n_invalid) *n_invalid = bad;
    return 0;
}
