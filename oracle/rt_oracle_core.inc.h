/*
 * rt_oracle_core.inc.h — CPU ORACLE core (test infrastructure, NOT product code).
 * Included twice by rt_oracle.c: once with RTO_FMA 0 (suffix _host) and once with RTO_FMA 1 (suffix _dev).
 *
 * Every float expression is written in ONE explicit form, FMA(a,b,c):
 *   RTO_FMA 0:  (a*b)+c with two roundings   == what g++ emits for the reference headers on x86-64
 *                                               (no FMA contraction; SURVEY A.4 host build);
 *   RTO_FMA 1:  fmaf(a,b,c), one rounding    == what nvcc+ptxas emit for the reference on sm_100.
 * The placement of each FMA was read off the reference's SASS (`cuobjdump -sass` of main.cu built with
 * `nvcc -O3 -arch=sm_100`): ptxas fuses every add/sub that has a product operand; when both operands
 * are products the LEFT one is fused and the right one is rounded:
 *     a*b + c*d  -> fma(a,b, c*d)          x - a*b -> fma(-a,b,x)        a*b - c*d -> fma(a,b,-(c*d))
 *     dot(v,w)   -> fma(vz,wz, fma(vx,wx, vy*wy))                      (vec3.h:91-93)
 * Division and sqrt are IEEE-correct on both (nvcc default -prec-div/-prec-sqrt).
 * This translation unit must be compiled with -ffp-contract=off.
 */

#if RTO_FMA
#define FMA(a, b, c) fmaf((a), (b), (c))
#define SUF(name) name##_dev
#else
#define FMA(a, b, c) (((a) * (b)) + (c))
#define SUF(name) name##_host
#endif

/* vec3.h:91-93 dot(); contraction pattern above */
static inline float SUF(dot3)(v3 a, v3 b) { return FMA(a.z, b.z, FMA(a.x, b.x, a.y * b.y)); }
/* vec3.h:34 length(), :146-148 unit_vector(): true divides */
static inline v3 SUF(unit_vector)(v3 v) {
    float len = sqrtf(SUF(dot3)(v, v));
    return V3(v.x / len, v.y / len, v.z / len);
}

/* sphere.h:17-46 sphere::hit.  Returns 1 and fills t (p, normal are derived by the caller only for
 * the final closest hit: they depend on nothing but t, the ray and the sphere). */
static inline int SUF(sphere_hit)(const rto_sphere *s, v3 o, v3 d, float t_min, float t_max, float *t_out,
                                  rto_counters *ctr) {
    ctr->sphere_tests++;
    v3 oc = V3(o.x - s->cx, o.y - s->cy, o.z - s->cz);            /* sphere.h:18 */
    float a = SUF(dot3)(d, d);                                     /* :19 */
    float b = SUF(dot3)(oc, d);                                    /* :20 */
    float c = FMA(-s->radius, s->radius, SUF(dot3)(oc, oc));       /* :21  dot(oc,oc) - r*r */
    float disc = FMA(b, b, -(a * c));                              /* :22  b*b - a*c */
    if (disc > 0.0f) {
        float sq = sqrtf(disc);
        float temp = (-b - sq) / a;                                /* :27 */
        if (temp < t_max && temp > t_min) { *t_out = temp; return 1; }
        temp = (-b + sq) / a;                                      /* :36 */
        if (temp < t_max && temp > t_min) { *t_out = temp; return 1; }
    }
    return 0;
}

/* sphere.h:30-33: rec.p = A + t*B (ray.h:13), rec.normal = (p - center) / radius */
static inline void SUF(hit_point)(const rto_sphere *s, v3 o, v3 d, float t, v3 *p, v3 *n) {
    *p = V3(FMA(d.x, t, o.x), FMA(d.y, t, o.y), FMA(d.z, t, o.z));
    *n = V3((p->x - s->cx) / s->radius, (p->y - s->cy) / s->radius, (p->z - s->cz) / s->radius);
}

/* hitable_list.h:16-31: linear closest hit, strict '<' against closest_so_far */
static int SUF(hit_list)(const rto_sphere *sph, int n, v3 o, v3 d, float t_min, float t_max, float *t_hit,
                         rto_counters *ctr) {
    int best = -1;
    float closest = t_max;
    for (int i = 0; i < n; i++) {
        float t;
        if (sph[i].mat == RTO_MAT_NONE) continue;   /* SURVEY D3: undefined slots never hit */
        if (SUF(sphere_hit)(&sph[i], o, d, t_min, closest, &t, ctr)) { best = i; closest = t; }
    }
    *t_hit = closest;
    return best;
}

/* acceleration_structure.h:226-244 intersect_ray_aabb: slab test of the infinite line, float divides,
 * no FMA opportunity (sub then div).  NaN comparisons are false exactly as in the reference. */
static inline int SUF(ray_aabb)(v3 o, v3 d, const float *bx, rto_counters *ctr) {
    ctr->aabb_tests++;
    float tmin = (bx[0] - o.x) / d.x, tmax = (bx[3] - o.x) / d.x;
    if (tmin > tmax) { float t = tmin; tmin = tmax; tmax = t; }
    float tymin = (bx[1] - o.y) / d.y, tymax = (bx[4] - o.y) / d.y;
    if (tymin > tymax) { float t = tymin; tymin = tymax; tymax = t; }
    if ((tmin > tymax) || (tymin > tmax)) return 0;
    if (tymin > tmin) tmin = tymin;
    if (tymax < tmax) tmax = tymax;
    float tzmin = (bx[2] - o.z) / d.z, tzmax = (bx[5] - o.z) / d.z;
    if (tzmin > tzmax) { float t = tzmin; tzmin = tzmax; tzmax = t; }
    if ((tmin > tzmax) || (tzmin > tmax)) return 0;
    return 1;
}

typedef struct { int best; float closest; } SUF(phit);

/* acceleration_structure.h:276-304 traverseTree (recursive, fixed child order, no pruning) with
 * processHit (:254-265) inlined */
static void SUF(traverse)(const oct_view *ov, const rto_sphere *sph, v3 o, v3 d, int node, SUF(phit) *res,
                          rto_counters *ctr) {
    const int32_t *nd = oct_node(ov, node);
    if (!SUF(ray_aabb)(o, d, (const float *)(nd + 1), ctr)) return;
    const int32_t *children = nd + 7;
    if (nd[0] == RTO_TREE_HEIGHT) {
        for (int i = 0; i < 8; i++) {
            int leaf = children[i];
            if (leaf == 0) return;
            if (leaf >= ov->leaf_count) return;              /* :286-289 */
            const int32_t *lf = oct_leaf(ov, leaf);
            int cnt = lf[ov->spl];
            for (int j = 0; j < cnt; j++) {
                int idx = lf[j];
                if (idx == 0) continue;                      /* :255 */
                if (sph[idx].mat == RTO_MAT_NONE) continue;  /* SURVEY D3 */
                float t;
                if (SUF(sphere_hit)(&sph[idx], o, d, 0.001f, res->closest, &t, ctr)) {
                    res->best = idx; res->closest = t;
                }
            }
        }
        return;
    }
    for (int i = 0; i < 8; i++)
        if (children[i] != 0) SUF(traverse)(ov, sph, o, d, children[i], res, ctr);
}

/* acceleration_structure.h:319-342 hitTree: ground sphere (index 0) first, then the tree.  The reference's slot 0 is always the
 * ground; a caller's world may leave it undefined, and an undefined slot is never hit (SURVEY D3), here as in the flat list. */
static int SUF(hit_tree)(const oct_view *ov, const rto_sphere *sph, v3 o, v3 d, float *t_hit, rto_counters *ctr) {
    SUF(phit) res = {-1, FLT_MAX};
    float t;
    if (sph[0].mat != RTO_MAT_NONE && SUF(sphere_hit)(&sph[0], o, d, 0.001f, FLT_MAX, &t, ctr)) { res.best = 0; res.closest = t; }
    SUF(traverse)(ov, sph, o, d, 0, &res, ctr);
    *t_hit = res.closest;
    return res.best;
}

/* material.h:33-41 random_in_unit_sphere; RANDVEC3 draws left to right on the device (SURVEY D4) */
static inline v3 SUF(random_in_unit_sphere)(xorwow *rng) {
    v3 p;
    do {
        float u0 = xorwow_uniform(rng), u1 = xorwow_uniform(rng), u2 = xorwow_uniform(rng);
        p = V3(FMA(u0, 2.0f, -1.0f), FMA(u1, 2.0f, -1.0f), FMA(u2, 2.0f, -1.0f)); /* 2*v - (1,1,1) */
    } while (SUF(dot3)(p, p) >= 1.0f);
    return p;
}

/* material.h:43-45 reflect: v - 2*dot(v,n)*n */
static inline v3 SUF(reflect)(v3 v, v3 n) {
    float d2 = 2.0f * SUF(dot3)(v, n);
    return V3(FMA(-n.x, d2, v.x), FMA(-n.y, d2, v.y), FMA(-n.z, d2, v.z));
}

/* material.h:17-31 refract */
static inline int SUF(refract)(v3 v, v3 n, float ni_over_nt, v3 *refracted) {
    v3 uv = SUF(unit_vector)(v);
    float dt = SUF(dot3)(uv, n);
    float disc = FMA(-(ni_over_nt * ni_over_nt), FMA(-dt, dt, 1.0f), 1.0f);  /* 1 - ni*ni*(1 - dt*dt) */
    if (disc > 0.0f) {
        float sq = sqrtf(disc);
        /* ni*(uv - n*dt) - n*sqrt(disc) */
        refracted->x = FMA(sq, -n.x, ni_over_nt * FMA(dt, -n.x, uv.x));
        refracted->y = FMA(sq, -n.y, ni_over_nt * FMA(dt, -n.y, uv.y));
        refracted->z = FMA(sq, -n.z, ni_over_nt * FMA(dt, -n.z, uv.z));
        return 1;
    }
    return 0;
}

/* material.h:11-15 schlick; pow is computed in 32 bit (powf) */
static inline float SUF(schlick)(float cosine, float ref_idx) {
    float r0 = (1.0f - ref_idx) / (1.0f + ref_idx);
    r0 = r0 * r0;
    return FMA(1.0f - r0, powf(1.0f - cosine, 5.0f), r0);
}

/* material.h:55-60 / :68-73 / :81-113.  Returns 0 when the ray is absorbed (metal only). */
static int SUF(scatter)(const rto_sphere *s, v3 d_in, v3 p, v3 n, v3 *atten, v3 *d_out, xorwow *rng) {
    if (s->mat == RTO_MAT_LAMBERTIAN) {
        v3 r = SUF(random_in_unit_sphere)(rng);
        /* target = p + normal + r ; direction = target - p (SURVEY D12: not simplified) */
        v3 target = V3((p.x + n.x) + r.x, (p.y + n.y) + r.y, (p.z + n.z) + r.z);
        *d_out = V3(target.x - p.x, target.y - p.y, target.z - p.z);
        *atten = V3(s->ax, s->ay, s->az);
        return 1;
    }
    if (s->mat == RTO_MAT_METAL) {
        v3 refl = SUF(reflect)(SUF(unit_vector)(d_in), n);
        v3 r = SUF(random_in_unit_sphere)(rng);        /* drawn even when fuzz == 0 */
        *d_out = V3(FMA(s->param, r.x, refl.x), FMA(s->param, r.y, refl.y), FMA(s->param, r.z, refl.z));
        *atten = V3(s->ax, s->ay, s->az);
        return SUF(dot3)(*d_out, n) > 0.0f;
    }
    /* dielectric */
    {
        float ref_idx = s->param;
        v3 outward, refracted = V3(0, 0, 0);
        v3 reflected = SUF(reflect)(d_in, n);
        float ni_over_nt, reflect_prob, cosine;
        *atten = V3(1.0f, 1.0f, 1.0f);
        float ddn = SUF(dot3)(d_in, n);
        if (ddn > 0.0f) {
            outward = V3(-n.x, -n.y, -n.z);
            ni_over_nt = ref_idx;
            cosine = ddn / sqrtf(SUF(dot3)(d_in, d_in));
            cosine = sqrtf(FMA(-(ref_idx * ref_idx), FMA(-cosine, cosine, 1.0f), 1.0f));
        } else {
            outward = n;
            ni_over_nt = 1.0f / ref_idx;
            cosine = -ddn / sqrtf(SUF(dot3)(d_in, d_in));
        }
        if (SUF(refract)(d_in, outward, ni_over_nt, &refracted))
            reflect_prob = SUF(schlick)(cosine, ref_idx);
        else {
            reflect_prob = 1.0f;
#if RTO_FMA
            /* material.h:88 leaves `refracted` UNINITIALISED and material.h:109 reads it when total internal reflection meets
             * curand_uniform == 1.0 (the draw is in (0, 1]; p ~ 3e-8 per such event; BASELINE config 3 at full size has one:
             * pixel (2070, 687), sample 36).  What the reference's sm_100 build then uses is whatever its registers hold — read off
             * the SASS of `render` (cuobjdump, nvcc 12.9 -O3 -arch=sm_100; dielectric::scatter at 0x4f10, the select at 0x6c90):
             * refracted = (R16, R2, R17) = (v.y, v.z, unit_vector(v).y), v = r_in.direction().  The host build of the reference
             * leaves other garbage there; this oracle's host mode keeps zero. */
            refracted = V3(d_in.y, d_in.z, d_in.y / sqrtf(SUF(dot3)(d_in, d_in)));
#endif
        }
        if (xorwow_uniform(rng) < reflect_prob) *d_out = reflected;
        else *d_out = refracted;
        return 1;
    }
}

/* camera.h:12-18 random_in_unit_disk + :45-49 get_ray */
static inline void SUF(get_ray)(const rto_camera *c, float s, float t, xorwow *rng, v3 *o, v3 *d) {
    float px, py;
    do {
        float u0 = xorwow_uniform(rng), u1 = xorwow_uniform(rng);
        px = FMA(u0, 2.0f, -1.0f);
        py = FMA(u1, 2.0f, -1.0f);
    } while (FMA(px, px, py * py) >= 1.0f);                 /* dot(p,p) with p.z == 0 */
    float rdx = c->lens_radius * px, rdy = c->lens_radius * py;
    float off[3], org[3], dir[3];
    for (int k = 0; k < 3; k++) {
        off[k] = FMA(c->u[k], rdx, c->v[k] * rdy);          /* u*rd.x + v*rd.y */
        org[k] = c->origin[k] + off[k];
        /* lower_left_corner + s*horizontal + t*vertical - origin - offset */
        dir[k] = (FMA(c->vertical[k], t, FMA(c->horizontal[k], s, c->lower_left_corner[k])) - c->origin[k]) - off[k];
    }
    *o = V3(org[0], org[1], org[2]);
    *d = V3(dir[0], dir[1], dir[2]);
}

/* main.cu:43-75 color() */
static v3 SUF(color)(const rto_sphere *sph, int n, const oct_view *ov, int use_octree, int max_depth, v3 o, v3 d,
                     xorwow *rng, rto_counters *ctr, uint32_t *depth_out) {
    v3 att = V3(1.0f, 1.0f, 1.0f);
    for (int i = 0; i < max_depth; i++) {
        float t;
        int idx;
        ctr->rays++;
        *depth_out = (uint32_t)(i + 1);
        if (use_octree) idx = SUF(hit_tree)(ov, sph, o, d, &t, ctr);
        else idx = SUF(hit_list)(sph, n, o, d, 0.001f, FLT_MAX, &t, ctr);
        if (idx >= 0) {
            v3 p, nrm, a, dn;
            SUF(hit_point)(&sph[idx], o, d, t, &p, &nrm);
            if (SUF(scatter)(&sph[idx], d, p, nrm, &a, &dn, rng)) {
                att = V3(att.x * a.x, att.y * a.y, att.z * a.z);
                o = p; d = dn;
            } else {
                return V3(0, 0, 0);
            }
        } else {
            v3 ud = SUF(unit_vector)(d);
            float t2 = 0.5f * (ud.y + 1.0f);
            float omt = 1.0f - t2;
            /* (1-t)*(1,1,1) + t*(0.5,0.7,1.0) */
            v3 c = V3(FMA(t2, 0.5f, omt), FMA(t2, 0.7f, omt), t2 + omt);
            return V3(att.x * c.x, att.y * c.y, att.z * c.z);
        }
    }
    return V3(0, 0, 0);
}

/* main.cu:96-117 render(): one pixel, ns samples chained through one XORWOW state (SURVEY D8) */
static void SUF(render_pixel)(const rto_sphere *sph, int n, const rto_camera *cam, const oct_view *ov,
                              const rto_render_params *p, int i, int j, float *fb_gamma, float *fb_linear,
                              rto_counters *ctr) {
    int pixel_index = j * p->nx + i;
    xorwow rng;
    if (p->seed_mode == RTO_SEED_UPSTREAM) xorwow_init_subseq(&rng, 1984, (uint64_t)pixel_index);   /* main.cu:90 (commented out at HEAD) */
    else xorwow_init(&rng, (uint64_t)(int64_t)(1984 + pixel_index));                                /* main.cu:93 */
    v3 col = V3(0, 0, 0);
    for (int s = 0; s < p->ns; s++) {
        float u = ((float)i + xorwow_uniform(&rng)) / (float)p->nx;   /* main.cu:104 */
        float v = ((float)j + xorwow_uniform(&rng)) / (float)p->ny;   /* main.cu:105 */
        v3 o, d;
        uint32_t depth = 0;
        SUF(get_ray)(cam, u, v, &rng, &o, &d);
        v3 c = SUF(color)(sph, n, ov, p->use_octree, p->max_depth, o, d, &rng, ctr, &depth);
        col = V3(col.x + c.x, col.y + c.y, col.z + c.z);
        ctr->paths++;
        if (depth > ctr->max_depth) ctr->max_depth = depth;
    }
    if (fb_linear) {
        fb_linear[3 * pixel_index + 0] = col.x;
        fb_linear[3 * pixel_index + 1] = col.y;
        fb_linear[3 * pixel_index + 2] = col.z;
    }
    if (fb_gamma) {
        float k = (float)(1.0 / (double)(float)p->ns);               /* vec3.h:137-144: k = 1.0/t */
        fb_gamma[3 * pixel_index + 0] = sqrtf(col.x * k);            /* main.cu:111-114 */
        fb_gamma[3 * pixel_index + 1] = sqrtf(col.y * k);
        fb_gamma[3 * pixel_index + 2] = sqrtf(col.z * k);
    }
}

static int SUF(closest_hit)(const rto_sphere *sph, int n, const oct_view *ov, int use_octree, v3 o, v3 d,
                            float *t_out) {
    rto_counters ctr;
    memset(&ctr, 0, sizeof ctr);
    return use_octree ? SUF(hit_tree)(ov, sph, o, d, t_out, &ctr)
                      : SUF(hit_list)(sph, n, o, d, 0.001f, FLT_MAX, t_out, &ctr);
}

#undef FMA
#undef SUF
