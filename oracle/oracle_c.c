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
