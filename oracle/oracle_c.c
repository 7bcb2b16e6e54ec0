/* ORACLE -- TEST INFRASTRUCTURE ONLY (never linked into the product library).
 *
 * Plain-C restatement of the scalar / integer pieces of the hot path, used where the torch-based
 * oracle (sapcu_oracle.py) would be too slow or too memory hungry (large kNN checks) and as an
 * independent second statement of the neuron recurrences.  Pinned against tests/golden/ by
 * tests/test_oracle_golden.py.  Build: `make -C oracle` -> oracle/_build/liboracle_c.so.
 * Compile WITHOUT -ffast-math / FMA contraction (-ffp-contract=off): operation order matters.
 */
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

/* KDTree(data).query(seeds, K)[1] (reference generation.py:110,127,153) as an exact fp64 brute force:
 * reduced distance ((dx*dx)+(dy*dy))+(dz*dz); ascending, ties -> lowest index (insertion into a sorted list). */
void oracle_knn_f64(const double* cloud, int64_t n, const double* seeds, int64_t s, int k, int32_t* idx) {
    double* bd = (double*)malloc(sizeof(double) * (size_t)k);
    for (int64_t q = 0; q < s; ++q) {
        int cnt = 0;
        int32_t* bi = idx + q * k;
        for (int64_t p = 0; p < n; ++p) {
            const double dx = cloud[3 * p] - seeds[3 * q], dy = cloud[3 * p + 1] - seeds[3 * q + 1],
                         dz = cloud[3 * p + 2] - seeds[3 * q + 2];
            const double d = ((dx * dx) + (dy * dy)) + (dz * dz);
            if (cnt == k && !(d < bd[k - 1])) continue;      /* equal distance, larger index: stays out */
            int pos = cnt < k ? cnt : k - 1;
            while (pos > 0 && d < bd[pos - 1]) { bd[pos] = bd[pos - 1]; bi[pos] = bi[pos - 1]; --pos; }
            bd[pos] = d; bi[pos] = (int32_t)p;
            if (cnt < k) ++cnt;
        }
    }
    free(bd);
}

/* farthest_point_sample (reference generate.py:56-74) in fp32 from any start index: running distances 1e32, squared
 * distance (dx*dx + dy*dy) + dz*dz, `dist < distance` update, arg-max with the first maximum (lowest index). */
void oracle_fps_f32(const float* xyz, int64_t n, int64_t npoint, int64_t start, int64_t* out) {
    float* dist = (float*)malloc(sizeof(float) * (size_t)n);
    for (int64_t i = 0; i < n; ++i) dist[i] = 1e32f;
    int64_t far = start;
    for (int64_t it = 0; it < npoint; ++it) {
        out[it] = far;
        const float cx = xyz[3 * far], cy = xyz[3 * far + 1], cz = xyz[3 * far + 2];
        int64_t best = 0;
        float bd = -1.0f;
        for (int64_t p = 0; p < n; ++p) {
            const float dx = xyz[3 * p] - cx, dy = xyz[3 * p + 1] - cy, dz = xyz[3 * p + 2] - cz;
            const float d = (dx * dx + dy * dy) + dz * dz;
            if (d < dist[p]) dist[p] = d;
            if (dist[p] > bd) { bd = dist[p]; best = p; }
        }
        far = best;
    }
    free(dist);
}

static float clampf(float v, float lo, float hi) { return fminf(fmaxf(v, lo), hi); }

/* eval-mode soft spike (reference fn/snn_coder.py:135-153) */
static float spike_fn(float v) {
    const float vc = clampf(v, -10.0f, 10.0f);
    const float g = expf(-(vc * vc) / 2.0f) / 2.5066282746310002f;
    const float sg = 1.0f / (1.0f + expf(-(10.0f * vc)));
    return 0.5f * g + 0.5f * sg;
}

/* T fed-back steps of the LIF (eif == NULL) or EIF neuron from the zero state
 * (reference fn/snn_coder.py:109-133, fd/snn_coder.py:223-261).
 * x [rows][C]; prm [4][C] RAW (unclamped) {decay, adapt, refr, theta0}; eif [2][C] RAW {delta_T, theta_rh};
 * out [T][rows][C]. */
void oracle_neuron_chain(const float* x, int64_t rows, int C, int T, const float* prm, const float* eif, float* out) {
    for (int64_t r = 0; r < rows; ++r)
        for (int c = 0; c < C; ++c) {
            const float d = clampf(prm[c], 0.1f, 0.99f), a = clampf(prm[C + c], 0.001f, 0.1f),
                        rr = clampf(prm[2 * C + c], 0.1f, 0.95f), th0 = prm[3 * C + c];
            float dT = 0.f, thrh = 0.f;
            if (eif) { dT = clampf(eif[c], 0.1f, 5.0f); thrh = clampf(eif[C + c], 0.1f, 2.0f); }
            float m = 0.f, th = th0, rho = 0.f, s = x[r * C + c];
            for (int t = 0; t < T; ++t) {
                float ex = 0.f;
                if (eif) ex = dT * expf(clampf((m - thrh) / (dT + 1e-6f), -5.0f, 5.0f));
                float in = s * (rho <= 0.f ? 1.0f : 0.0f);
                m = m * d * (1.0f - rho) + in;
                if (eif) m = m + ex;
                s = spike_fn(m - th);
                m = m * (1.0f - s);
                rho = rho * rr + s;
                th = th + a * s;
                th = th0 + (th - th0) * 0.95f;
                out[((int64_t)t * rows + r) * C + c] = s;
            }
        }
}

/* rotation_matrix_from_vectors(n, [1,0,0]) (reference generation.py:30-47): n float32, result float64 row-major */
void oracle_rotation_to_x(const float* n, double* R) {
    /* np.linalg.norm(float32[3]) = sqrt(x.dot(x)): OpenBLAS sdot rounds each product to fp32 and accumulates in
     * double (measured: bit-exact on 20000 random vectors), then the sum is rounded back to fp32 */
    const float p0 = n[0] * n[0], p1 = n[1] * n[1], p2 = n[2] * n[2];
    const float nn = sqrtf((float)(((double)p0 + (double)p1) + (double)p2));
    const double a0 = (double)(n[0] / nn), a1 = (double)(n[1] / nn), a2 = (double)(n[2] / nn);
    const double v[3] = {0.0, a2, -a1};
    memset(R, 0, 9 * sizeof(double));
    R[0] = R[4] = R[8] = 1.0;
    if (v[1] == 0.0 && v[2] == 0.0) return;
    const double c = a0, s = sqrt((v[0] * v[0] + v[1] * v[1]) + v[2] * v[2]);
    const double K[3][3] = {{0.0, -v[2], v[1]}, {v[2], 0.0, -v[0]}, {-v[1], v[0], 0.0}};
    const double f = (1.0 - c) / (s * s);
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
            const double k2 = (K[i][0] * K[0][j] + K[i][1] * K[1][j]) + K[i][2] * K[2][j];
            R[3 * i + j] = (R[3 * i + j] + K[i][j]) + k2 * f;
        }
}

/* data[idx] - seed, optional rotation, cast to float (reference generation.py:128-129,154-160,137) */
void oracle_gather_center_rotate(const double* cloud, const double* seeds, const int32_t* idx, int64_t s, int k,
                                 const float* normals, float* patches) {
    for (int64_t q = 0; q < s; ++q) {
        double R[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
        if (normals) oracle_rotation_to_x(normals + 3 * q, R);
        for (int j = 0; j < k; ++j) {
            const int64_t p = idx[q * k + j];
            const double d[3] = {cloud[3 * p] - seeds[3 * q], cloud[3 * p + 1] - seeds[3 * q + 1], cloud[3 * p + 2] - seeds[3 * q + 2]};
            for (int r = 0; r < 3; ++r) {
                const double o = normals ? (R[3 * r] * d[0] + R[3 * r + 1] * d[1]) + R[3 * r + 2] * d[2] : d[r];
                patches[(q * k + j) * 3 + r] = (float)o;
            }
        }
    }
}

/* seed + (double)(n * d) (reference generation.py:171-172) */
void oracle_displace(const double* seeds, const float* normals, const float* dist, int64_t s, double* out) {
    for (int64_t i = 0; i < 3 * s; ++i) out[i] = seeds[i] + (double)(normals[i] * dist[i / 3]);
}

/* ------------------------------------------------------------------------------------------------------------------
 * Seed generator (dense.cpp:175-252 as specified in the header of csrc/seedgen.cu), restated as the reference's plain
 * FIFO flood fill: one queue, one pop at a time, a hash set of evaluated voxel ids.  Nothing here shares the device's
 * level / keep-first claim / scan structure; the only thing taken over is the arithmetic, in the same operation order. */

typedef struct { double x, y, z; } v3;
static v3 v3sub(v3 a, v3 b) { v3 r = {a.x - b.x, a.y - b.y, a.z - b.z}; return r; }
static v3 v3add(v3 a, v3 b) { v3 r = {a.x + b.x, a.y + b.y, a.z + b.z}; return r; }
static v3 v3mul(v3 a, double s) { v3 r = {a.x * s, a.y * s, a.z * s}; return r; }
static v3 v3div(v3 a, double s) { v3 r = {a.x / s, a.y / s, a.z / s}; return r; }
static double v3dot(v3 a, v3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
static v3 v3cross(v3 a, v3 b) { v3 r = {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; return r; }
static double v3dist(v3 a, v3 b) {
    return sqrt((a.x - b.x) * (a.x - b.x) + (a.y - b.y) * (a.y - b.y) + (a.z - b.z) * (a.z - b.z));
}

/* closest point on triangle abc to p: dense.cpp:135-174, branch for branch (csrc/geom.cuh point_tri) */
static v3 point_tri(v3 a, v3 b, v3 c, v3 p) {
    const v3 ab = v3sub(b, a), ac = v3sub(c, a), bc = v3sub(c, b);
    const double snom = v3dot(v3sub(p, a), ab), sdenom = v3dot(v3sub(p, b), v3sub(a, b));
    const double tnom = v3dot(v3sub(p, a), ac), tdenom = v3dot(v3sub(p, c), v3sub(a, c));
    if (snom <= 0.0 && tnom <= 0.0) return a;
    const double unom = v3dot(v3sub(p, b), bc), udenom = v3dot(v3sub(p, c), v3sub(b, c));
    if (sdenom <= 0.0 && unom <= 0.0) return b;
    if (tdenom <= 0.0 && udenom <= 0.0) return c;
    const v3 n = v3cross(v3sub(b, a), v3sub(c, a));
    const double vc = v3dot(n, v3cross(v3sub(a, p), v3sub(b, p)));
    if (vc <= 0.0 && snom >= 0.0 && sdenom >= 0.0) return v3add(a, v3div(v3mul(ab, snom), snom + sdenom));
    const double va = v3dot(n, v3cross(v3sub(b, p), v3sub(c, p)));
    if (va <= 0.0 && unom >= 0.0 && udenom >= 0.0) return v3add(b, v3div(v3mul(bc, unom), unom + udenom));
    const double vb = v3dot(n, v3cross(v3sub(c, p), v3sub(a, p)));
    if (vb <= 0.0 && tnom >= 0.0 && tdenom >= 0.0) return v3add(a, v3div(v3mul(ac, tnom), tnom + tdenom));
    const double u = va / (va + vb + vc);
    const double v = vb / (va + vb + vc);
    const double w = 1.0 - u - v;
    return v3add(v3add(v3mul(a, u), v3mul(b, v)), v3mul(c, w));
}

/* open-addressing set of int voxel ids (any int, negative ones included) */
typedef struct { int32_t* key; uint8_t* used; int64_t cap, n; } idset;
static uint64_t id_hash(int32_t id) {
    uint64_t h = (uint64_t)(uint32_t)id * 0x9E3779B97F4A7C15ull;
    return h ^ (h >> 29);
}
static int idset_init(idset* s, int64_t cap) {
    s->cap = cap; s->n = 0;
    s->key = (int32_t*)malloc(sizeof(int32_t) * (size_t)cap);
    s->used = (uint8_t*)calloc((size_t)cap, 1);
    return s->key && s->used ? 0 : -1;
}
static int64_t idset_slot(const idset* s, int32_t id) {
    int64_t i = (int64_t)(id_hash(id) & (uint64_t)(s->cap - 1));
    while (s->used[i] && s->key[i] != id) i = (i + 1) & (s->cap - 1);
    return i;
}
/* 1 if id was new (and is now in the set), 0 if present, -1 on allocation failure */
static int idset_add(idset* s, int32_t id) {
    if (2 * (s->n + 1) > s->cap) {
        idset t;
        if (idset_init(&t, 2 * s->cap)) return -1;
        for (int64_t i = 0; i < s->cap; ++i)
            if (s->used[i]) { const int64_t j = idset_slot(&t, s->key[i]); t.used[j] = 1; t.key[j] = s->key[i]; }
        t.n = s->n;
        free(s->key); free(s->used);
        *s = t;
    }
    const int64_t i = idset_slot(s, id);
    if (s->used[i]) return 0;
    s->used[i] = 1; s->key[i] = id; ++s->n;
    return 1;
}

/* uniform grid over the (N + quirk) search points for the exact 10-NN */
typedef struct { double org[3], g; int dim[3]; int64_t* start; int32_t* item; } pgrid;
static int pgrid_cell(const pgrid* G, int a, double v) {
    const double f = floor((v - G->org[a]) / G->g);
    return f < 0 ? 0 : (f >= G->dim[a] ? G->dim[a] - 1 : (int)f);
}
static int pgrid_build(pgrid* G, const double* P, int64_t n) {
    double lo[3] = {P[0], P[1], P[2]}, hi[3] = {P[0], P[1], P[2]}, ext = 0.0;
    for (int64_t i = 1; i < n; ++i)
        for (int a = 0; a < 3; ++a) { lo[a] = fmin(lo[a], P[3 * i + a]); hi[a] = fmax(hi[a], P[3 * i + a]); }
    for (int a = 0; a < 3; ++a) ext = fmax(ext, hi[a] - lo[a]);
    const int side = (int)fmin(128.0, ceil(cbrt((double)n)));
    G->g = ext > 0.0 ? ext / side : 1.0;
    int64_t ncell = 1;
    for (int a = 0; a < 3; ++a) {
        G->org[a] = lo[a];
        G->dim[a] = (int)fmin((double)side, floor((hi[a] - lo[a]) / G->g) + 1.0);
        ncell *= G->dim[a];
    }
    G->start = (int64_t*)calloc((size_t)ncell + 1, sizeof(int64_t));
    G->item = (int32_t*)malloc(sizeof(int32_t) * (size_t)n);
    int64_t* cid = (int64_t*)malloc(sizeof(int64_t) * (size_t)n);
    if (!G->start || !G->item || !cid) { free(cid); return -1; }
    for (int64_t i = 0; i < n; ++i) {
        cid[i] = ((int64_t)pgrid_cell(G, 0, P[3 * i]) * G->dim[1] + pgrid_cell(G, 1, P[3 * i + 1])) * G->dim[2] +
                 pgrid_cell(G, 2, P[3 * i + 2]);
        ++G->start[cid[i] + 1];
    }
    for (int64_t c = 0; c < ncell; ++c) G->start[c + 1] += G->start[c];
    int64_t* fill = (int64_t*)malloc(sizeof(int64_t) * (size_t)ncell);
    if (!fill) { free(cid); return -1; }
    memcpy(fill, G->start, sizeof(int64_t) * (size_t)ncell);
    for (int64_t i = 0; i < n; ++i) G->item[fill[cid[i]]++] = (int32_t)i;
    free(fill); free(cid);
    return 0;
}

/* the 10 points nearest to c in (d, index) order, d = (dx*dx + dy*dy) + dz*dz with (p - c): the order the device's
 * strict-`<` insertion in index order produces.  Ring r of grid cells is searched until no point outside the visited
 * block can be closer than the 10th distance (with a relative margin far above the rounding of d). */
static void knn10(const pgrid* G, const double* P, v3 c, double* bd, int32_t* bi) {
    for (int k = 0; k < 10; ++k) { bd[k] = INFINITY; bi[k] = -1; }
    const double q[3] = {c.x, c.y, c.z};
    int ci[3];
    for (int a = 0; a < 3; ++a) ci[a] = pgrid_cell(G, a, q[a]);
    for (int r = 0;; ++r) {
        const int x0 = ci[0] - r < 0 ? 0 : ci[0] - r, x1 = ci[0] + r < G->dim[0] ? ci[0] + r : G->dim[0] - 1;
        const int y0 = ci[1] - r < 0 ? 0 : ci[1] - r, y1 = ci[1] + r < G->dim[1] ? ci[1] + r : G->dim[1] - 1;
        const int z0 = ci[2] - r < 0 ? 0 : ci[2] - r, z1 = ci[2] + r < G->dim[2] ? ci[2] + r : G->dim[2] - 1;
        for (int x = x0; x <= x1; ++x) {
            for (int y = y0; y <= y1; ++y) {
                const int full = abs(x - ci[0]) == r || abs(y - ci[1]) == r;     /* else only the two z caps */
                const int zstep = full || r == 0 ? 1 : 2 * r;
                for (int z = full ? z0 : ci[2] - r; z <= (full ? z1 : ci[2] + r); z += zstep) {
                    if (z < 0 || z >= G->dim[2]) continue;
                    const int64_t cell = ((int64_t)x * G->dim[1] + y) * G->dim[2] + z;
                    for (int64_t t = G->start[cell]; t < G->start[cell + 1]; ++t) {
                        const int32_t j = G->item[t];
                        const double dx = P[3 * j] - c.x, dy = P[3 * j + 1] - c.y, dz = P[3 * j + 2] - c.z;
                        const double d = (dx * dx + dy * dy) + dz * dz;
                        if (!(d < bd[9] || (d == bd[9] && j < bi[9]))) continue;
                        int k = 9;
                        while (k > 0 && (d < bd[k - 1] || (d == bd[k - 1] && j < bi[k - 1]))) {
                            bd[k] = bd[k - 1]; bi[k] = bi[k - 1]; --k;
                        }
                        bd[k] = d; bi[k] = j;
                    }
                }
            }
        }
        /* lower bound on the distance of every point in a cell outside the block |cell - ci| <= r */
        double lb = INFINITY;
        for (int a = 0; a < 3; ++a) {
            if (ci[a] - r - 1 >= 0) lb = fmin(lb, q[a] - (G->org[a] + (ci[a] - r) * G->g));
            if (ci[a] + r + 1 < G->dim[a]) lb = fmin(lb, (G->org[a] + (ci[a] + r + 1) * G->g) - q[a]);
        }
        if (lb == INFINITY) return;                                            /* every cell visited */
        if (lb > 0.0 && lb * lb * (1.0 - 1e-9) > bd[9]) return;
    }
}

static v3 voxel_center(int id, int B, double cell) {
    int t = id;
    const int z = t % B; t /= B;
    const int y = t % B; t /= B;
    const int x = t;
    v3 r = {x * cell + 0.5 * cell - 0.5, y * cell + 0.5 * cell - 0.5, z * cell + 0.5 * cell - 0.5};
    return r;
}

/* fprintf("%lf") (dense.cpp:232) read back as a double (generation.py's np.loadtxt) */
static double text_round6(double v) {
    char buf[64];
    snprintf(buf, sizeof buf, "%lf", v);
    return strtod(buf, NULL);
}

void oracle_round6_text(const double* v, int64_t n, double* out) {
    for (int64_t i = 0; i < n; ++i) out[i] = text_round6(v[i]);
}

/* int voxel-id arithmetic with the two's-complement wrap of the device's int */
static int32_t id_of(int x, int y, int z, int B) {
    return (int32_t)((uint32_t)x * (uint32_t)B * (uint32_t)B + (uint32_t)y * (uint32_t)B + (uint32_t)z);
}

/* Seeds of cloud [N][3] at voxel size `cell`, in emission order; the first `cap` are stored in out [cap][3], the total
 * goes to *count.  level_stats (may be NULL) receives, per BFS level L < max_levels, {queue entries of level L,
 * 6 * voxels of level L that expand}; the second number is the length of level L + 1.  Returns the number of levels,
 * or -1 if memory ran out. */
int64_t oracle_seedgen(const double* cloud, int64_t N, double cell, int quirk_origin, int round6, double* out, int64_t cap,
                       int64_t* count, int64_t* level_stats, int64_t max_levels) {
    const int B = (int)round(1.0 / cell);
    const int64_t NT = N + (quirk_origin ? 1 : 0);
    double* P = (double*)calloc((size_t)NT * 3, sizeof(double));          /* the quirk point stays at the origin */
    int64_t qcap = N > 1024 ? N : 1024, head = 0, tail = 0;
    int32_t* queue = (int32_t*)malloc(sizeof(int32_t) * (size_t)qcap);
    pgrid G = {{0, 0, 0}, 0, {0, 0, 0}, NULL, NULL};
    idset seen = {NULL, NULL, 0, 0};
    int64_t levels = -1, emitted = 0;
    if (!P || !queue || idset_init(&seen, 1 << 16) || (memcpy(P, cloud, sizeof(double) * 3 * (size_t)N), pgrid_build(&G, P, NT)))
        goto done;
    /* initial queue: the voxel of every input point, in input order (dense.cpp:186-191) */
    for (int64_t i = 0; i < N; ++i) {
        const double v = floor((cloud[3 * i] + 0.5) / cell) * B * B + floor((cloud[3 * i + 1] + 0.5) / cell) * B +
                         floor((cloud[3 * i + 2] + 0.5) / cell);
        queue[tail++] = (int)v;
    }
    int64_t level = 0, level_end = tail, level_len = tail, expanding = 0;
    while (head < tail) {
        const int32_t id = queue[head++];
        const int fresh = idset_add(&seen, id);
        if (fresh < 0) goto done;
        if (fresh) {
            const v3 c = voxel_center(id, B, cell);
            double bd[10]; int32_t bi[10];
            knn10(&G, P, c, bd, bi);
            v3 p[10];                            /* p[9] nearest, p[8] second nearest; fewer than 10 points: origin */
            for (int k = 0; k < 10; ++k) {
                const int32_t j = bi[k];
                v3 t = {0.0, 0.0, 0.0};
                if (j >= 0 && j < N) { t.x = cloud[3 * j]; t.y = cloud[3 * j + 1]; t.z = cloud[3 * j + 2]; }
                p[9 - k] = t;
            }
            double td = 99999999999999.0;
            for (int k = 7; k >= 0; --k) {
                const double dd = v3dist(point_tri(p[k], p[8], p[9], c), c);
                if (dd < td) td = dd;
            }
            if (td >= 0.0110 && td <= 0.0150) {
                if (emitted < cap) {
                    v3 s = c;
                    if (round6) { s.x = text_round6(s.x); s.y = text_round6(s.y); s.z = text_round6(s.z); }
                    out[3 * emitted] = s.x; out[3 * emitted + 1] = s.y; out[3 * emitted + 2] = s.z;
                }
                ++emitted;
            }
            if (td <= 0.0150) {
                if (tail + 6 > qcap) {                                  /* compact, then grow */
                    memmove(queue, queue + head, sizeof(int32_t) * (size_t)(tail - head));
                    tail -= head; level_end -= head; head = 0;
                    if (tail + 6 > qcap / 2) {
                        int32_t* q2 = (int32_t*)realloc(queue, sizeof(int32_t) * (size_t)(2 * qcap));
                        if (!q2) goto done;
                        queue = q2; qcap *= 2;
                    }
                }
                int t = id;
                const int z = t % B; t /= B;
                const int y = t % B; t /= B;
                const int x = t;
                queue[tail++] = id_of(x + 1, y, z, B); queue[tail++] = id_of(x - 1, y, z, B);
                queue[tail++] = id_of(x, y + 1, z, B); queue[tail++] = id_of(x, y - 1, z, B);
                queue[tail++] = id_of(x, y, z + 1, B); queue[tail++] = id_of(x, y, z - 1, B);
                ++expanding;
            }
        }
        if (head == level_end) {                                        /* level L popped completely */
            if (level_stats && level < max_levels) { level_stats[2 * level] = level_len; level_stats[2 * level + 1] = 6 * expanding; }
            ++level;
            level_end = tail; level_len = tail - head; expanding = 0;
        }
    }
    levels = level;
    *count = emitted;
done:
    free(P); free(queue); free(G.start); free(G.item); free(seen.key); free(seen.used);
    return levels;
}
