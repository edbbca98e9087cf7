/* tests/oracle_hits.c — TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * The primary-hit buffers of tcrt_hit_buffers (include/tcrt.h) restated on the CPU with the pinned oracle's own code:
 * primary_ray, then nearest_hit (getCollision, RayTracer.cpp:50-89), then the n2 of build_hit (the CollisionObject's
 * normal ray, SceneObject.h:47-105).  oracle/tcrt_oracle.c is included unchanged, so these values are the ones its
 * renders (pinned to the reference) are built from.  Built by tests/test_hit_buffers.py with the oracle's flags:
 *   gcc -std=gnu11 -O2 -fPIC -shared -ffp-contract=off oracle_hits.c -lm
 */
#include "../oracle/tcrt_oracle.c"

/* Columns x0, x0+stride, ... < x1, x-major like frames: obj[k], dist[k], normal[3k..3k+2] for the k-th pixel.  A miss is
 * -1, far_dist, (+0, +0, +0).  Returns 0, or -1 on bad arguments. */
int tcrt_oracle_primary_hits(const tcrt_scene* s, const tcrt_camera* cam, const tcrt_params* p, int x0, int x1, int stride,
                             int* obj, float* dist, float* normal) {
    if (!s || !cam || !p || !obj || !dist || !normal || p->width <= 0 || p->height <= 0 || x0 < 0 || x1 > p->width ||
        x0 > x1 || stride < 1)
        return -1;
    oracle_counters c;
    memset(&c, 0, sizeof(c));
    g_cnt = &c;
    size_t k = 0;
    for (int x = x0; x < x1; x += stride)
        for (int z = 0; z < p->height; z++, k++) {
            v3 O, D;
            primary_ray(cam, p, x, z, &O, &D);
            float d, px, py, den;
            const int o = nearest_hit(s, p, O, D, &d, &px, &py, &den, &c);
            v3 n = v3_make(0.0f, 0.0f, 0.0f);
            if (o >= 0) {
                hit_record h;
                build_hit(s, o, d, px, py, den, O, D, &h);
                n = h.n2;
            }
            obj[k] = o;
            dist[k] = d;   /* nearest_hit leaves far_dist on a miss */
            normal[3 * k + 0] = n.x;
            normal[3 * k + 1] = n.y;
            normal[3 * k + 2] = n.z;
        }
    return 0;
}
