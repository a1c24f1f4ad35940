/* limu_oracle.c -- ORACLE: test infrastructure, not product code. See limu_oracle.h.
 *
 * Plain-C restatement of the reference hot path. "L/" = env_ws/src/limu of the reference.
 * Every per-point operation (voxel index, rigid transform, squared distance, gates) is written in the
 * reference's exact operation order so results are bit-identical to the compiled reference on
 * x86-64 without FMA contraction (build with -ffp-contract=off); pose-level algebra (exp/log/LDLT)
 * follows Sophus 1.22.10 / Eigen 3.4.0 and agrees to rounding.
 */
#include "limu_oracle.h"

#include <limits.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

/* ================================================================================================
 * Small vector helpers (operation orders pinned by tests/test_oracle_pin.py against Eigen 3.4.0 SSE2)
 * ============================================================================================== */

/* Eigen squaredNorm of a fixed 3-vector, SSE2 packet path: predux(packet(0,1)) then + element 2. */
static inline double sqn3(double a, double b, double c) { return (a * a + b * b) + c * c; }
/* Eigen squaredNorm of the 4 quaternion coefficients (x,y,z,w), two SSE2 packets: (x2+z2)+(y2+w2). */
static inline double sqn4(const double *q) { return (q[0] * q[0] + q[2] * q[2]) + (q[1] * q[1] + q[3] * q[3]); }

static inline void cross3(const double *a, const double *b, double *o) { /* Eigen cross3 */
    o[0] = a[1] * b[2] - a[2] * b[1];
    o[1] = a[2] * b[0] - a[0] * b[2];
    o[2] = a[0] * b[1] - a[1] * b[0];
}

/* Sophus SO3::operator*(point), sophus/so3.hpp:388-399: uv = qv x p; uv += uv; p + w*uv + qv x uv */
static inline void so3_rotate(const double *q, const double *p, double *o) {
    double uv[3], c[3];
    cross3(q, p, uv);
    uv[0] += uv[0]; uv[1] += uv[1]; uv[2] += uv[2];
    cross3(q, uv, c);
    o[0] = (p[0] + q[3] * uv[0]) + c[0];
    o[1] = (p[1] + q[3] * uv[1]) + c[1];
    o[2] = (p[2] + q[3] * uv[2]) + c[2];
}
/* Sophus SE3::operator*(point), sophus/se3.hpp:319-322: so3*p + t */
static inline void se3_apply(const double *T, const double *p, double *o) {
    double r[3];
    so3_rotate(T, p, r);
    o[0] = r[0] + T[4]; o[1] = r[1] + T[5]; o[2] = r[2] + T[6];
}
/* SO3(quaternion) constructor -> normalize(), sophus/so3.hpp:318-325 */
static inline void quat_normalize(double *q) {
    const double len = sqrt(sqn4(q));
    q[0] /= len; q[1] /= len; q[2] /= len; q[3] /= len;
}
/* sophus/so3.hpp:344-352 QuaternionProduct, then the normalising constructor (:358-369) */
static inline void so3_mul(const double *a, const double *b, double *o) {
    const double ax = a[0], ay = a[1], az = a[2], aw = a[3], bx = b[0], by = b[1], bz = b[2], bw = b[3];
    double r[4];
    r[3] = aw * bw - ax * bx - ay * by - az * bz;
    r[0] = aw * bx + ax * bw + ay * bz - az * by;
    r[1] = aw * by + ay * bw + az * bx - ax * bz;
    r[2] = aw * bz + az * bw + ax * by - ay * bx;
    quat_normalize(r);
    o[0] = r[0]; o[1] = r[1]; o[2] = r[2]; o[3] = r[3];
}

void lo_se3_mul(const double *a, const double *b, double *out) { /* se3.hpp:302-307 */
    double q[4], r[3];
    so3_mul(a, b, q);
    so3_rotate(a, b + 4, r);
    const double t0 = a[4] + r[0], t1 = a[5] + r[1], t2 = a[6] + r[2];
    out[0] = q[0]; out[1] = q[1]; out[2] = q[2]; out[3] = q[3];
    out[4] = t0; out[5] = t1; out[6] = t2;
}
void lo_se3_inv(const double *a, double *out) { /* se3.hpp:222-225, so3.hpp:246-248 */
    double q[4] = {-a[0], -a[1], -a[2], a[3]};
    quat_normalize(q);
    const double nt[3] = {a[4] * -1.0, a[5] * -1.0, a[6] * -1.0};
    double r[3];
    so3_rotate(q, nt, r);
    out[0] = q[0]; out[1] = q[1]; out[2] = q[2]; out[3] = q[3];
    out[4] = r[0]; out[5] = r[1]; out[6] = r[2];
}

#define SOPHUS_EPS 1e-10 /* sophus/common.hpp:157 */

static void hat3(const double *w, double *O) { /* so3.hpp:783-792, row-major 3x3 */
    O[0] = 0; O[1] = -w[2]; O[2] = w[1];
    O[3] = w[2]; O[4] = 0; O[5] = -w[0];
    O[6] = -w[1]; O[7] = w[0]; O[8] = 0;
}
/* Eigen 3.4.0 fixed 3x3 lazy products under SSE2 (column-major, 2-double packets): rows 0-1 of each
 * column go through the packet path, sum_k in order ((k0 + k1) + k2); row 2 goes through the scalar
 * redux unroller, which splits 3 terms as k0 + (k1 + k2). Pinned by tests/test_oracle_pin.py. */
static void mat3_mul(const double *A, const double *B, double *C) {
    for (int j = 0; j < 3; ++j) {
        for (int i = 0; i < 2; ++i)
            C[3 * i + j] = (A[3 * i] * B[j] + A[3 * i + 1] * B[3 + j]) + A[3 * i + 2] * B[6 + j];
        C[6 + j] = A[6] * B[j] + (A[7] * B[3 + j] + A[8] * B[6 + j]);
    }
}
static void mat3_vec(const double *A, const double *v, double *o) {
    for (int i = 0; i < 2; ++i) o[i] = (A[3 * i] * v[0] + A[3 * i + 1] * v[1]) + A[3 * i + 2] * v[2];
    o[2] = A[6] * v[0] + (A[7] * v[1] + A[8] * v[2]);
}

void lo_se3_exp(const double *a, double *out) { /* se3.hpp:852-861; so3.hpp:694-732, :550-571 */
    const double *ups = a, *om = a + 3;
    const double theta_sq = sqn3(om[0], om[1], om[2]);
    double theta, imag, real;
    if (theta_sq < SOPHUS_EPS * SOPHUS_EPS) {
        theta = 0.0;
        const double theta_po4 = theta_sq * theta_sq;
        imag = 0.5 - (1.0 / 48.0) * theta_sq + (1.0 / 3840.0) * theta_po4;
        real = 1.0 - (1.0 / 8.0) * theta_sq + (1.0 / 384.0) * theta_po4;
    } else {
        theta = sqrt(theta_sq);
        const double half = 0.5 * theta;
        imag = sin(half) / theta;
        real = cos(half);
    }
    out[3] = real; out[0] = imag * om[0]; out[1] = imag * om[1]; out[2] = imag * om[2];
    /* leftJacobian(omega, theta): theta_sq recomputed as theta*theta (so3.hpp:556) */
    const double tsq = theta * theta;
    double Om[9], Om2[9], V[9];
    hat3(om, Om);
    mat3_mul(Om, Om, Om2);
    static const double I3[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    if (tsq < SOPHUS_EPS * SOPHUS_EPS) {
        for (int i = 0; i < 9; ++i) V[i] = I3[i] + 0.5 * Om[i];
    } else {
        const double c1 = (1.0 - cos(theta)) / tsq, c2 = (theta - sin(theta)) / (tsq * theta);
        for (int i = 0; i < 9; ++i) V[i] = (I3[i] + c1 * Om[i]) + c2 * Om2[i];
    }
    mat3_vec(V, ups, out + 4);
}

void lo_se3_log(const double *T, double *x) { /* se3.hpp:237-253; so3.hpp:264-310, :573-597 */
    const double sqn = sqn3(T[0], T[1], T[2]), w = T[3];
    double two_atan, theta;
    if (sqn < SOPHUS_EPS * SOPHUS_EPS) {
        const double sw = w * w;
        two_atan = 2.0 / w - (2.0 / 3.0) * sqn / (w * sw);
        theta = 2.0 * sqn / w;
    } else {
        const double n = sqrt(sqn);
        const double at = (w < 0.0) ? atan2(-n, -w) : atan2(n, w);
        two_atan = 2.0 * at / n;
        theta = two_atan * n;
    }
    double om[3] = {two_atan * T[0], two_atan * T[1], two_atan * T[2]};
    const double tsq = theta * theta;
    double Om[9], Om2[9], Vi[9];
    hat3(om, Om);
    mat3_mul(Om, Om, Om2);
    static const double I3[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    if (tsq < SOPHUS_EPS * SOPHUS_EPS) {
        for (int i = 0; i < 9; ++i) Vi[i] = (I3[i] - 0.5 * Om[i]) + (1. / 12.) * Om2[i];
    } else {
        const double half = 0.5 * theta;
        const double c = (1.0 - 0.5 * theta * cos(half) / sin(half)) / (theta * theta);
        for (int i = 0; i < 9; ++i) Vi[i] = (I3[i] - 0.5 * Om[i]) + c * Om2[i];
    }
    mat3_vec(Vi, T + 4, x);
    x[3] = om[0]; x[4] = om[1]; x[5] = om[2];
}

void lo_delta_pose(const double *a, const double *b, double *x) { /* calculation_helpers.cpp:99-102 */
    double ai[7], d[7];
    lo_se3_inv(a, ai);
    lo_se3_mul(ai, b, d);
    lo_se3_log(d, x);
}

void lo_vox_index(const double *xyz, long n, double v, int *keys) { /* calculation_helpers.cpp:142-147 */
    for (long i = 0; i < 3 * n; ++i) keys[i] = (int)(xyz[i] / v);
}

void lo_transform(const double *T, double *xyz, long n) { /* calculation_helpers.cpp:121-133 */
    if (n <= 0) { printf("[INFO] utils::transform_points the points vector is empty\n"); return; }
    for (long i = 0; i < n; ++i) {
        double o[3];
        se3_apply(T, xyz + 3 * i, o);
        xyz[3 * i] = o[0]; xyz[3 * i + 1] = o[1]; xyz[3 * i + 2] = o[2];
    }
}

/* ================================================================================================
 * Voxel grid containers: insertion-ordered entries + open-addressing index on the full (i,j,k) key
 * ============================================================================================== */
typedef struct {
    int32_t *slot; /* entry index + 1; 0 empty; -1 tombstone */
    long n_slots, n_used;
} lo_index;

static inline uint64_t key_hash(const int *k) {
    uint64_t h = (uint64_t)(uint32_t)k[0] * 0x9E3779B185EBCA87ull;
    h ^= (uint64_t)(uint32_t)k[1] * 0xC2B2AE3D27D4EB4Full;
    h ^= (uint64_t)(uint32_t)k[2] * 0x165667B19E3779F9ull;
    h ^= h >> 29; h *= 0xBF58476D1CE4E5B9ull; h ^= h >> 32;
    return h;
}

struct lo_map {
    double vox_size, max_distance;
    int cap;
    int icp_mode;  /* 0 = the reference's neighbour rule; bit 0 (LO_ICP_NN27) = nearest point of the 27-cell neighbourhood (SURVEY 8f N2) */
    long n_entries, n_alive, entries_cap;
    int *keys;     /* 3 per entry (creation order) */
    int *counts;   /* points stored; -1 = erased entry */
    double *pts;   /* cap*3 per entry */
    lo_index ix;
};

static void index_rebuild(lo_map *m, long want) {
    long ns = 16;
    while (ns < want) ns <<= 1;
    free(m->ix.slot);
    m->ix.slot = (int32_t *)calloc((size_t)ns, sizeof(int32_t));
    m->ix.n_slots = ns; m->ix.n_used = 0;
    for (long e = 0; e < m->n_entries; ++e) {
        if (m->counts[e] < 0) continue;
        long s = (long)(key_hash(m->keys + 3 * e) & (uint64_t)(ns - 1));
        while (m->ix.slot[s] != 0) s = (s + 1) & (ns - 1);
        m->ix.slot[s] = (int32_t)(e + 1);
        ++m->ix.n_used;
    }
}
static long map_find(const lo_map *m, const int *k) {
    if (m->ix.n_slots == 0) return -1;
    const long mask = m->ix.n_slots - 1;
    long s = (long)(key_hash(k) & (uint64_t)mask);
    for (;;) {
        const int32_t v = m->ix.slot[s];
        if (v == 0) return -1;
        if (v > 0) {
            const int *kk = m->keys + 3 * (long)(v - 1);
            if (kk[0] == k[0] && kk[1] == k[1] && kk[2] == k[2]) return v - 1;
        }
        s = (s + 1) & mask;
    }
}
static long map_emplace(lo_map *m, const int *k) {
    if ((m->ix.n_used + 1) * 2 > m->ix.n_slots) index_rebuild(m, (m->n_alive + 1) * 4);
    if (m->n_entries == m->entries_cap) {
        m->entries_cap = m->entries_cap ? m->entries_cap * 2 : 1024;
        m->keys = (int *)realloc(m->keys, sizeof(int) * 3 * (size_t)m->entries_cap);
        m->counts = (int *)realloc(m->counts, sizeof(int) * (size_t)m->entries_cap);
        m->pts = (double *)realloc(m->pts, sizeof(double) * 3 * (size_t)m->cap * (size_t)m->entries_cap);
    }
    const long e = m->n_entries++;
    m->keys[3 * e] = k[0]; m->keys[3 * e + 1] = k[1]; m->keys[3 * e + 2] = k[2];
    m->counts[e] = 0;
    const long mask = m->ix.n_slots - 1;
    long s = (long)(key_hash(k) & (uint64_t)mask);
    while (m->ix.slot[s] != 0) s = (s + 1) & mask;
    m->ix.slot[s] = (int32_t)(e + 1);
    ++m->ix.n_used; ++m->n_alive;
    return e;
}
static void map_erase(lo_map *m, long e) {
    const long mask = m->ix.n_slots - 1;
    long s = (long)(key_hash(m->keys + 3 * e) & (uint64_t)mask);
    while (m->ix.slot[s] != (int32_t)(e + 1)) s = (s + 1) & mask;
    m->ix.slot[s] = -1;
    m->counts[e] = -1;
    --m->n_alive;
}

lo_map *lo_map_create(double vox_size, double max_distance, int cap) {
    lo_map *m = (lo_map *)calloc(1, sizeof(lo_map));
    m->vox_size = vox_size; m->max_distance = max_distance; m->cap = cap;
    return m;
}
void lo_map_clear(lo_map *m) {
    free(m->keys); free(m->counts); free(m->pts); free(m->ix.slot);
    m->keys = NULL; m->counts = NULL; m->pts = NULL; m->ix.slot = NULL;
    m->n_entries = m->n_alive = m->entries_cap = 0; m->ix.n_slots = m->ix.n_used = 0;
}
void lo_map_destroy(lo_map *m) { if (m) { lo_map_clear(m); free(m); } }
int lo_map_empty(const lo_map *m) { return m->n_alive == 0; }
long lo_map_num_voxels(const lo_map *m) { return m->n_alive; }

/* insert_points, voxel_hash_map.cpp:12-62 + VoxelBlock::add_point voxel_block.cpp:68-73: points are
 * appended in input order until max_points_per_voxel; later ones are dropped. */
void lo_map_insert(lo_map *m, const double *xyz, long n) {
    for (long i = 0; i < n; ++i) {
        int k[3];
        lo_vox_index(xyz + 3 * i, 1, m->vox_size, k);
        long e = map_find(m, k);
        if (e < 0) e = map_emplace(m, k);
        if (m->counts[e] < m->cap) {
            double *d = m->pts + 3 * ((size_t)e * (size_t)m->cap + (size_t)m->counts[e]);
            d[0] = xyz[3 * i]; d[1] = xyz[3 * i + 1]; d[2] = xyz[3 * i + 2];
            ++m->counts[e];
        }
    }
}

/* remove_points_from_far, voxel_hash_map.cpp:146-171, as it executes under null locks: for every voxel
 * whose INDEX distance^2 to the origin's voxel exceeds max_distance^2 (units as written, :148,160),
 * drop its points farther than max_distance (metres) from origin (voxel_block.cpp:107-118, order
 * preserving), and erase the voxel if it became empty. */
void lo_map_remove_far(lo_map *m, const double *origin) {
    const double max_dist_sq = m->max_distance * m->max_distance;
    int ov[3];
    lo_vox_index(origin, 1, m->vox_size, ov);
    for (long e = 0; e < m->n_entries; ++e) {
        if (m->counts[e] < 0) continue;
        const int *k = m->keys + 3 * e;
        /* Vector3i squaredNorm: int arithmetic, which wraps modulo 2^32 in the reference's build; written unsigned so that the wrap is
         * defined behaviour here rather than signed overflow */
        const uint32_t dx = (uint32_t)k[0] - (uint32_t)ov[0], dy = (uint32_t)k[1] - (uint32_t)ov[1], dz = (uint32_t)k[2] - (uint32_t)ov[2];
        const int d2 = (int)(dx * dx + dy * dy + dz * dz);
        if ((double)d2 > max_dist_sq) {
            double *p = m->pts + 3 * (size_t)e * (size_t)m->cap;
            int w = 0;
            for (int r = 0; r < m->counts[e]; ++r) {
                const double ax = p[3 * r] - origin[0], ay = p[3 * r + 1] - origin[1], az = p[3 * r + 2] - origin[2];
                if (!(sqn3(ax, ay, az) > max_dist_sq)) {
                    p[3 * w] = p[3 * r]; p[3 * w + 1] = p[3 * r + 1]; p[3 * w + 2] = p[3 * r + 2];
                    ++w;
                }
            }
            m->counts[e] = w;
            if (w == 0) map_erase(m, e);
        }
    }
}

void lo_map_update(lo_map *m, const double *xyz, long n, const double *pose7) { /* :132-144 */
    double *w = (double *)malloc(sizeof(double) * 3 * (size_t)(n > 0 ? n : 1));
    memcpy(w, xyz, sizeof(double) * 3 * (size_t)n);
    lo_transform(pose7, w, n);
    lo_map_insert(m, w, n);
    lo_map_remove_far(m, pose7 + 4);
    free(w);
}

/* VoxelBlock::get_closest_point, voxel_block.cpp:87-105: strict '<', first minimum wins. */
static int block_closest(const lo_map *m, long e, const double *p) {
    const double *b = m->pts + 3 * (size_t)e * (size_t)m->cap;
    int best = -1;
    double min_dist = 1.7976931348623157e308;
    for (int r = 0; r < m->counts[e]; ++r) {
        const double d = sqn3(p[0] - b[3 * r], p[1] - b[3 * r + 1], p[2] - b[3 * r + 2]);
        if (d < min_dist) { best = r; min_dist = d; }
    }
    return best;
}

/* get_closest_neighbour, voxel_hash_map.cpp:64-102.
 * (a) own voxel present -> closest point inside it only;
 * (b) else among the 27 cells around it, the TOP of a max-heap on (index distance^2, block address):
 *     the farthest occupied cell, ties to the higher address == later-created voxel (shim definition);
 * (c) none -> (0,0,0). */
static long closest_entry(const lo_map *m, const double *p) {
    int k[3];
    lo_vox_index(p, 1, m->vox_size, k);
    long e = map_find(m, k);
    if (e >= 0) return e;
    long best = -1;
    int best_d = -1;
    for (int i = k[0] - 1; i <= k[0] + 1; ++i)
        for (int j = k[1] - 1; j <= k[1] + 1; ++j)
            for (int l = k[2] - 1; l <= k[2] + 1; ++l) {
                const int q[3] = {i, j, l};
                const long c = map_find(m, q);
                if (c < 0) continue;
                const int dx = k[0] - i, dy = k[1] - j, dz = k[2] - l;
                const int d = dx * dx + dy * dy + dz * dz;
                if (d > best_d || (d == best_d && c > best)) { best_d = d; best = c; }
            }
    return best;
}

/* Opt-in neighbour rule LO_ICP_NN27 (SURVEY section 8f N2; NOT in the reference -- this restatement is the definition the CUDA path is
 * checked against): the nearest stored point over all 27 cells around the query's voxel, cells visited x-outermost, points in storage
 * order, strict '<' (first minimum wins); nothing stored there -> no match, i.e. (0,0,0) like rule (c). */
static long closest27_entry(const lo_map *m, const double *p, int *rank_out) {
    int k[3];
    lo_vox_index(p, 1, m->vox_size, k);
    long best = -1;
    double min_dist = 1.7976931348623157e308;
    *rank_out = -1;
    for (int i = k[0] - 1; i <= k[0] + 1; ++i)
        for (int j = k[1] - 1; j <= k[1] + 1; ++j)
            for (int l = k[2] - 1; l <= k[2] + 1; ++l) {
                const int q[3] = {i, j, l};
                const long c = map_find(m, q);
                if (c < 0) continue;
                const double *b = m->pts + 3 * (size_t)c * (size_t)m->cap;
                for (int r = 0; r < m->counts[c]; ++r) {
                    const double d = sqn3(p[0] - b[3 * r], p[1] - b[3 * r + 1], p[2] - b[3 * r + 2]);
                    if (d < min_dist) { min_dist = d; best = c; *rank_out = r; }
                }
            }
    return best;
}
void lo_map_set_mode(lo_map *m, int icp_mode) { m->icp_mode = icp_mode; }

void lo_map_closest(const lo_map *m, const double *xyz, long n, double *out, int *out_key, int *out_rank) {
    for (long i = 0; i < n; ++i) {
        const double *p = xyz + 3 * i;
        int r = -1;
        long e;
        if (m->icp_mode & 1) e = closest27_entry(m, p, &r);
        else {
            e = closest_entry(m, p);
            if (e >= 0) r = block_closest(m, e, p);
        }
        if (e >= 0 && r >= 0) {
            const double *t = m->pts + 3 * ((size_t)e * (size_t)m->cap + (size_t)r);
            out[3 * i] = t[0]; out[3 * i + 1] = t[1]; out[3 * i + 2] = t[2];
            if (out_key) { out_key[3 * i] = m->keys[3 * e]; out_key[3 * i + 1] = m->keys[3 * e + 1]; out_key[3 * i + 2] = m->keys[3 * e + 2]; }
        } else {
            out[3 * i] = out[3 * i + 1] = out[3 * i + 2] = 0.0;
            if (out_key) out_key[3 * i] = out_key[3 * i + 1] = out_key[3 * i + 2] = INT_MIN;
        }
        if (out_rank) out_rank[i] = r;
    }
}

long lo_map_correspondences(const lo_map *m, const double *xyz, long n, double tau, double *src, double *tgt, long *out_idx) {
    const double max_sq = tau * tau; /* :112 */
    long c = 0;
    for (long i = 0; i < n; ++i) {
        double f[3];
        lo_map_closest(m, xyz + 3 * i, 1, f, NULL, NULL);
        const double *p = xyz + 3 * i;
        if (sqn3(f[0] - p[0], f[1] - p[1], f[2] - p[2]) < max_sq) { /* (found - point).squaredNorm() :120 */
            if (src) { src[3 * c] = p[0]; src[3 * c + 1] = p[1]; src[3 * c + 2] = p[2]; }
            if (tgt) { tgt[3 * c] = f[0]; tgt[3 * c + 1] = f[1]; tgt[3 * c + 2] = f[2]; }
            if (out_idx) out_idx[c] = i;
            ++c;
        }
    }
    return c;
}

long lo_map_dump(const lo_map *m, int *keys, int *counts, double *pts, long max_vox, long max_pts, long *n_pts) {
    long nv = 0, np = 0;
    for (long e = 0; e < m->n_entries; ++e) {
        if (m->counts[e] < 0) continue;
        if (nv < max_vox) {
            if (keys) { keys[3 * nv] = m->keys[3 * e]; keys[3 * nv + 1] = m->keys[3 * e + 1]; keys[3 * nv + 2] = m->keys[3 * e + 2]; }
            if (counts) counts[nv] = m->counts[e];
        }
        for (int r = 0; r < m->counts[e]; ++r) {
            if (pts && np < max_pts) memcpy(pts + 3 * np, m->pts + 3 * ((size_t)e * (size_t)m->cap + (size_t)r), 3 * sizeof(double));
            ++np;
        }
        ++nv;
    }
    if (n_pts) *n_pts = np;
    return nv;
}

/* ================================================================================================
 * Registration: helpers/registration.cpp
 * ============================================================================================== */

/* Eigen 3.4.0 LDLT (Cholesky/LDLT.h:300-395 factorisation with diagonal pivoting, :569-607 solve),
 * 6x6, lower triangle, in place. Solves A x = b. */
static void ldlt6_solve(const double *Ain, const double *b, double *x) {
    enum { N = 6 };
    double A[N][N];
    int tr[N];
    for (int i = 0; i < N; ++i) for (int j = 0; j < N; ++j) A[i][j] = Ain[N * i + j];
    double temp[N];
    int zero_diag = 0;
    for (int k = 0; k < N; ++k) {
        int big = k;
        double bigv = fabs(A[k][k]);
        for (int i = k + 1; i < N; ++i) if (fabs(A[i][i]) > bigv) { bigv = fabs(A[i][i]); big = i; }
        tr[k] = big;
        if (k != big) {
            const int s = N - big - 1;
            for (int c = 0; c < k; ++c) { double t = A[k][c]; A[k][c] = A[big][c]; A[big][c] = t; }
            for (int r = 0; r < s; ++r) { double t = A[N - s + r][k]; A[N - s + r][k] = A[N - s + r][big]; A[N - s + r][big] = t; }
            { double t = A[k][k]; A[k][k] = A[big][big]; A[big][big] = t; }
            for (int i = k + 1; i < big; ++i) { double t = A[i][k]; A[i][k] = A[big][i]; A[big][i] = t; }
        }
        const int rs = N - k - 1;
        if (k > 0) {
            for (int c = 0; c < k; ++c) temp[c] = A[c][c] * A[k][c];
            double acc = 0.0;
            for (int c = 0; c < k; ++c) acc += A[k][c] * temp[c];
            A[k][k] -= acc;
            for (int r = 0; r < rs; ++r) {
                double a2 = 0.0;
                for (int c = 0; c < k; ++c) a2 += A[k + 1 + r][c] * temp[c];
                A[k + 1 + r][k] -= a2;
            }
        }
        const double akk = A[k][k];
        const int valid = fabs(akk) > 0.0;
        if (k == 0 && !valid) { for (int j = 0; j < N; ++j) tr[j] = j; zero_diag = 1; break; }
        if (rs > 0 && valid) for (int r = 0; r < rs; ++r) A[k + 1 + r][k] /= akk;
    }
    (void)zero_diag;
    double d[N];
    for (int i = 0; i < N; ++i) d[i] = b[i];
    for (int k = 0; k < N; ++k) if (tr[k] != k) { double t = d[k]; d[k] = d[tr[k]]; d[tr[k]] = t; }
    for (int i = 0; i < N; ++i) for (int c = 0; c < i; ++c) d[i] -= A[i][c] * d[c];       /* unit-lower forward */
    for (int i = 0; i < N; ++i) { if (fabs(A[i][i]) > 2.2250738585072014e-308) d[i] /= A[i][i]; else d[i] = 0.0; }
    for (int i = N - 1; i >= 0; --i) for (int c = i + 1; c < N; ++c) d[i] -= A[c][i] * d[c]; /* L^T backward */
    for (int k = N - 1; k >= 0; --k) if (tr[k] != k) { double t = d[k]; d[k] = d[tr[k]]; d[tr[k]] = t; }
    for (int i = 0; i < N; ++i) x[i] = d[i];
}

/* align_clouds, registration.cpp:43-92. J = [I3 | -hat(s)] (:46-54), w = th^2/(th+|r|^2)^2 (:57-58),
 * H += J^T w J, g += J^T w r (:75-76), x = LDLT(H).solve(-g) (:90), exp(x) (:91). */
void lo_align(const double *src, const double *tgt, long n, double th, double *H36, double *g6, double *x6, double *pose7) {
    double H[36], g[6];
    memset(H, 0, sizeof H); memset(g, 0, sizeof g);
    for (long i = 0; i < n; ++i) {
        const double *s = src + 3 * i, *t = tgt + 3 * i;
        const double r[3] = {s[0] - t[0], s[1] - t[1], s[2] - t[2]};
        double J[3][6] = {{1, 0, 0, 0, s[2], -s[1]}, {0, 1, 0, -s[2], 0, s[0]}, {0, 0, 1, s[1], -s[0], 0}};
        const double res_sq = sqn3(r[0], r[1], r[2]);
        const double w = (th * th) / ((th + res_sq) * (th + res_sq));
        for (int a = 0; a < 6; ++a) {
            const double ja0 = J[0][a] * w, ja1 = J[1][a] * w, ja2 = J[2][a] * w;
            for (int b = 0; b < 6; ++b) H[6 * a + b] += (ja0 * J[0][b] + ja1 * J[1][b]) + ja2 * J[2][b];
            g[a] += (ja0 * r[0] + ja1 * r[1]) + ja2 * r[2];
        }
    }
    double ng[6], x[6];
    for (int i = 0; i < 6; ++i) ng[i] = -g[i];
    ldlt6_solve(H, ng, x);
    if (H36) memcpy(H36, H, sizeof H);
    if (g6) memcpy(g6, g, sizeof g);
    if (x6) memcpy(x6, x, sizeof x);
    if (pose7) lo_se3_exp(x, pose7);
}

/* ---- opt-in point-to-plane residual LO_ICP_PLANE (SURVEY section 8f N2; NOT in the reference: this restatement is the definition) ----
 * Plane of a correspondence = the plane of the matched point's VOXEL: with c >= 5 stored points, mean mu and scatter S = sum (p-mu)(p-mu)^T,
 * the normal is the eigenvector of S's smallest eigenvalue, found by 5 cyclic Jacobi sweeps (rotations (0,1), (0,2), (1,2); only + - * /
 * sqrt, so the device reproduces it bit for bit). The voxel is planar when l_min <= 0.04 l_mid (thickness <= 0.2 x the minor in-plane
 * spread; line-like and blob-like voxels are rejected) and its correspondences are dropped otherwise, as are voxels with < 5 points.
 * Residual e = n.(s - t), weight w = th^2/(th + e^2)^2, Jacobian row a = [n ; s x n] in the reference's perturbation model
 * (s' = exp(x) s, J_point = [I | -hat(s)], registration.cpp:46-54), H += w a a^T, g += w a e, x = LDLT(H).solve(-g).
 * The solve carries a weak prior on the initial guess (the motion model's prediction), as the measurement update of a LiDAR-inertial
 * filter does: with xi = log(T_icp), the correction accumulated so far, x = LDLT(H + D).solve(-(g + D xi)),
 * D = diag(mu, mu, mu, mu rho^2, mu rho^2, mu rho^2), mu = LO_PLANE_PRIOR = 1 (one unit-weight correspondence per axis),
 * rho^2 = LO_PLANE_PRIOR_ARM2 = 100 m^2 (a 10 m lever arm for the rotational part). Against the thousands of correspondences of a
 * populated map D is negligible (the bias is ~1e-3 of a centimetre-sized correction); but a map of ONE scan with small voxels offers a
 * keypoint cloud only 1..40 planar voxels, H (rank <= that number, far less when they share a normal) does not determine six degrees of
 * freedom, and the unregularised step ran away by up to 20 m on scan 1 in 7 of 60 random point-to-plane configurations -- in this
 * restatement and on the device alike (profiles/r2_random_campaign.json). Directions the planes do not observe stay at the prediction.
 * (A prior on the STEP instead -- fixed Levenberg-Marquardt damping -- also stops the runaway but creeps along those directions for
 * hundreds of iterations before the twist falls below the convergence threshold.) */
#define LO_PLANE_MIN_POINTS 5
#define LO_PLANE_RATIO 0.04
#define LO_PLANE_PRIOR 1.0
#define LO_PLANE_PRIOR_ARM2 100.0
int lo_plane_normal(const double *b, int c, double *nrm) {   /* b: c points, array-of-structs */
    if (c < LO_PLANE_MIN_POINTS) return 0;
    double mu[3] = {0, 0, 0};
    for (int r = 0; r < c; ++r) { mu[0] += b[3 * r]; mu[1] += b[3 * r + 1]; mu[2] += b[3 * r + 2]; }
    mu[0] /= (double)c; mu[1] /= (double)c; mu[2] /= (double)c;
    double A[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}}, V[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
    for (int r = 0; r < c; ++r) {
        const double dx = b[3 * r] - mu[0], dy = b[3 * r + 1] - mu[1], dz = b[3 * r + 2] - mu[2];
        A[0][0] += dx * dx; A[0][1] += dx * dy; A[0][2] += dx * dz; A[1][1] += dy * dy; A[1][2] += dy * dz; A[2][2] += dz * dz;
    }
    A[1][0] = A[0][1]; A[2][0] = A[0][2]; A[2][1] = A[1][2];
    static const int PQ[3][2] = {{0, 1}, {0, 2}, {1, 2}};
    for (int sweep = 0; sweep < 5; ++sweep)
        for (int k = 0; k < 3; ++k) {
            const int p = PQ[k][0], q = PQ[k][1];
            const double apq = A[p][q];
            if (apq == 0.0) continue;
            const double theta = (A[q][q] - A[p][p]) / (2.0 * apq);
            const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
            const double cs = 1.0 / sqrt(t * t + 1.0), sn = t * cs;
            const int o = 3 - p - q;                     /* the third index */
            const double app = A[p][p], aqq = A[q][q], aop = A[o][p], aoq = A[o][q];
            A[p][p] = app - t * apq; A[q][q] = aqq + t * apq; A[p][q] = A[q][p] = 0.0;
            A[o][p] = A[p][o] = cs * aop - sn * aoq;
            A[o][q] = A[q][o] = sn * aop + cs * aoq;
            for (int i = 0; i < 3; ++i) { const double vip = V[i][p], viq = V[i][q]; V[i][p] = cs * vip - sn * viq; V[i][q] = sn * vip + cs * viq; }
        }
    int lo = 0;
    if (A[1][1] < A[lo][lo]) lo = 1;
    if (A[2][2] < A[lo][lo]) lo = 2;
    const int i1 = (lo + 1) % 3, i2 = (lo + 2) % 3;
    const double mid = A[i1][i1] < A[i2][i2] ? A[i1][i1] : A[i2][i2];
    if (!(mid > 0.0) || !(A[lo][lo] <= LO_PLANE_RATIO * mid)) return 0;
    nrm[0] = V[0][lo]; nrm[1] = V[1][lo]; nrm[2] = V[2][lo];
    return 1;
}
static int voxel_normal(const lo_map *m, long e, double *nrm) {
    return lo_plane_normal(m->pts + 3 * (size_t)e * (size_t)m->cap, m->counts[e], nrm);
}

/* One Gauss-Newton step of the point-to-plane variant over the current source cloud. Returns the number of plane correspondences. */
static long plane_step(const lo_map *m, const double *source, long n, double tau, double th, double *H, double *g) {
    memset(H, 0, 36 * sizeof(double)); memset(g, 0, 6 * sizeof(double));
    const double max_sq = tau * tau;
    long used = 0;
    for (long i = 0; i < n; ++i) {
        const double *s = source + 3 * i;
        double t[3];
        int key[3], rank;
        lo_map_closest(m, s, 1, t, key, &rank);
        if (rank < 0) continue;
        if (!(sqn3(t[0] - s[0], t[1] - s[1], t[2] - s[2]) < max_sq)) continue;
        double nr[3];
        if (!voxel_normal(m, map_find(m, key), nr)) continue;
        const double e = (nr[0] * (s[0] - t[0]) + nr[1] * (s[1] - t[1])) + nr[2] * (s[2] - t[2]);
        const double den = th + e * e;
        const double w = (th * th) / (den * den);
        const double a[6] = {nr[0], nr[1], nr[2], s[1] * nr[2] - s[2] * nr[1], s[2] * nr[0] - s[0] * nr[2], s[0] * nr[1] - s[1] * nr[0]};
        for (int r = 0; r < 6; ++r) {
            const double wa = w * a[r];
            for (int c = 0; c < 6; ++c) H[6 * r + c] += wa * a[c];
            g[r] += wa * e;
        }
        ++used;
    }
    return used;
}

static double norm6(const double *x) { /* Eigen norm() of a 6-vector, SSE2: 3 packets then predux */
    const double a = (x[0] * x[0] + x[2] * x[2]) + x[4] * x[4];
    const double b = (x[1] * x[1] + x[3] * x[3]) + x[5] * x[5];
    return sqrt(a + b);
}

/* ICP, registration.cpp:94-130. */
int lo_icp(const lo_map *m, const double *xyz, long n, const double *init7, double tau, double th, int max_iter,
           double eps, double *pose7, double *est_trace, long *ncorr_trace, double *hg_trace, double *src_after) {
    if (lo_map_empty(m)) { memcpy(pose7, init7, 7 * sizeof(double)); return 0; } /* :99-100 */
    const size_t bytes = sizeof(double) * 3 * (size_t)(n > 0 ? n : 1);
    double *source = (double *)malloc(bytes), *cs = (double *)malloc(bytes), *ct = (double *)malloc(bytes);
    memcpy(source, xyz, sizeof(double) * 3 * (size_t)n);
    lo_transform(init7, source, n);                                   /* :102-103 */
    double T_icp[7] = {0, 0, 0, 1, 0, 0, 0};                          /* :106 */
    int j = 0;
    for (; j < max_iter; ++j) {                                       /* :108 */
        long c;
        double est[7], H[36], g[6], lg[6], tmp[7];
        if (m->icp_mode & 2) {                                        /* opt-in point-to-plane variant (not in the reference) */
            double ng[6], x[6];
            c = plane_step(m, source, n, tau, th, H, g);
            double Hd[36], xi[6];
            memcpy(Hd, H, sizeof Hd);                                 /* (the trace keeps H and g without the prior) */
            lo_se3_log(T_icp, xi);
            for (int i = 0; i < 3; ++i) {
                Hd[7 * i] += LO_PLANE_PRIOR; Hd[7 * (i + 3)] += LO_PLANE_PRIOR * LO_PLANE_PRIOR_ARM2;
                ng[i] = -(g[i] + LO_PLANE_PRIOR * xi[i]);
                ng[i + 3] = -(g[i + 3] + (LO_PLANE_PRIOR * LO_PLANE_PRIOR_ARM2) * xi[i + 3]);
            }
            ldlt6_solve(Hd, ng, x);
            lo_se3_exp(x, est);
        } else {
            c = lo_map_correspondences(m, source, n, tau, cs, ct, NULL); /* :111 */
            lo_align(cs, ct, c, th, H, g, NULL, est);                 /* :116 */
        }
        lo_transform(est, source, n);                                 /* :119 */
        lo_se3_mul(est, T_icp, tmp); memcpy(T_icp, tmp, sizeof tmp);  /* :122 */
        if (est_trace) memcpy(est_trace + 7 * j, est, sizeof est);
        if (ncorr_trace) ncorr_trace[j] = c;
        if (hg_trace) { memcpy(hg_trace + 42 * j, H, sizeof H); memcpy(hg_trace + 42 * j + 36, g, sizeof g); }
        lo_se3_log(est, lg);
        if (norm6(lg) < eps) { ++j; break; }                          /* :124-125 */
    }
    lo_se3_mul(T_icp, init7, pose7);                                  /* :129 */
    if (src_after) memcpy(src_after, source, sizeof(double) * 3 * (size_t)n);
    free(source); free(cs); free(ct);
    return j;
}

/* ================================================================================================
 * Deskew: helpers/deskew.cpp:10-28
 * ============================================================================================== */
void lo_deskew(const float *xyz, const double *ts, long n, const double *T0, const double *T1, double *out) {
    double twist[6];
    lo_delta_pose(T0, T1, twist);                                     /* :14 */
    for (long i = 0; i < n; ++i) {
        const double p[3] = {(double)xyz[3 * i], (double)xyz[3 * i + 1], (double)xyz[3 * i + 2]};
        const double s = ts[i] - 0.5;                                 /* mid_pose_timestamp deskew.hpp:12 */
        const double st[6] = {s * twist[0], s * twist[1], s * twist[2], s * twist[3], s * twist[4], s * twist[5]};
        double M[7];
        lo_se3_exp(st, M);                                            /* :24 */
        se3_apply(M, p, out + 3 * i);                                 /* :25 */
    }
}

/* ================================================================================================
 * IMU-propagated backward deskew: kalman/ekf.cpp:420-468, kalman/helper.hpp:35-40
 * ============================================================================================== */
/* utils::ang_vel_to_rmat (helper.hpp:35-40): Eigen::AngleAxisd(dt*|w|, w.normalized()).toRotationMatrix()
 * (Eigen/src/Geometry/AngleAxis.h toRotationMatrix; normalized(): v / sqrt(squaredNorm) when squaredNorm > 0). */
static void ang_vel_to_rmat(const double *w, double dt, double *R) {
    const double z = sqn3(w[0], w[1], w[2]);
    const double nrm = sqrt(z);
    double ax[3] = {w[0], w[1], w[2]};
    if (z > 0.0) { ax[0] = w[0] / nrm; ax[1] = w[1] / nrm; ax[2] = w[2] / nrm; }
    const double angle = dt * nrm;
    const double s = sin(angle), c = cos(angle);
    const double sx = s * ax[0], sy = s * ax[1], sz = s * ax[2];
    const double cx = (1.0 - c) * ax[0], cy = (1.0 - c) * ax[1], cz = (1.0 - c) * ax[2];
    double tmp;
    tmp = cx * ax[1]; R[1] = tmp - sz; R[3] = tmp + sz;
    tmp = cx * ax[2]; R[2] = tmp + sy; R[6] = tmp - sy;
    tmp = cy * ax[2]; R[5] = tmp - sx; R[7] = tmp + sx;
    R[0] = cx * ax[0] + c; R[4] = cy * ax[1] + c; R[8] = cz * ax[2] + c;
}
void lo_deskew_imu(float *xyz, const float *curv_ms, long n, const double *table, long M, const double *rot_end, const double *pos_lidar_end,
                   const double *p_il, double *out) {
    long i = n - 1;
    for (long h = M - 2; h >= 0 && n > 0; --h) {                       /* it_kp = end-1 .. begin+1, head = *(it_kp-1) (:422-424) */
        const double *T = table + 22 * h;
        const double off = T[0], *acc = T + 1, *gyr = T + 4, *vel = T + 7, *pos = T + 10, *Rimu = T + 13;
        for (; (double)curv_ms[i] / 1000.0 > off; --i) {                /* :433 */
            const double dt = (double)curv_ms[i] / 1000.0 - off;        /* :435 */
            double Rw[9], Ri[9], t1[3], t2[3];
            ang_vel_to_rmat(gyr, dt, Rw);
            mat3_mul(Rimu, Rw, Ri);                                     /* R_i = R_imu * ang_vel_to_rmat(gyr, dt) :444 */
            mat3_vec(Ri, p_il, t1);
            double Tei[3];
            for (int a = 0; a < 3; ++a) Tei[a] = (((pos[a] + vel[a] * dt) + (0.5 * acc[a]) * (dt * dt)) + t1[a]) - pos_lidar_end[a];   /* :445 */
            const double P[3] = {(double)xyz[3 * i], (double)xyz[3 * i + 1], (double)xyz[3 * i + 2]};
            mat3_vec(Ri, P, t2);
            const double v[3] = {t2[0] + Tei[0], t2[1] + Tei[1], t2[2] + Tei[2]};
            for (int a = 0; a < 3; ++a)                                 /* rot_end^T * v :448, stored as float :451-453 */
                xyz[3 * i + a] = (float)((rot_end[a] * v[0] + rot_end[3 + a] * v[1]) + rot_end[6 + a] * v[2]);
            if (i == 0) break;                                          /* :455-456: the first point is NOT consumed, so every remaining
                                                                         * (older) head whose offset is below its time compensates it AGAIN */
        }
    }
    for (long k = 0; k < 3 * n; ++k) out[k] = (double)xyz[k];           /* :458-468 */
}

/* ================================================================================================
 * Downsampling and IQR: icp.cpp:9-30, :88-136, common.hpp:22-63
 * ============================================================================================== */
long lo_voxel_downsample(const double *xyz, long n, double s, double *out, long *out_idx) {
    lo_map *grid = lo_map_create(s, 0.0, 1);
    long c = 0;
    for (long i = 0; i < n; ++i) {
        int k[3];
        lo_vox_index(xyz + 3 * i, 1, s, k);
        if (map_find(grid, k) >= 0) continue;                         /* first point wins :16-18 */
        map_emplace(grid, k);
        if (out) memcpy(out + 3 * c, xyz + 3 * i, 3 * sizeof(double)); /* iteration order == insertion order */
        if (out_idx) out_idx[c] = i;
        ++c;
    }
    lo_map_destroy(grid);
    return c;
}

static int cmp_double(const void *a, const void *b) {
    const double x = *(const double *)a, y = *(const double *)b;
    return (x > y) - (x < y);
}
static double median_sorted(const double *a, long size) { /* common.hpp:22-38 on an already sorted range */
    const long half = size / 2;
    if (size % 2 == 0) return (a[half - 1] + a[half]) / 2.0;
    return a[half];
}
long lo_iqr(const double *xyz, long n, double *out, double *bounds2) {
    if (n <= 0) return 0; /* reference reads past an empty range here (UB); defined as empty output */
    double *d = (double *)malloc(sizeof(double) * (size_t)n), *a = (double *)malloc(sizeof(double) * (size_t)n);
    for (long i = 0; i < n; ++i) {
        const double x = xyz[3 * i], y = xyz[3 * i + 1], z = xyz[3 * i + 2];
        d[i] = x * x + y * y + z * z;                                 /* icp.cpp:97-100 */
    }
    memcpy(a, d, sizeof(double) * (size_t)n);
    qsort(a, (size_t)n, sizeof(double), cmp_double);
    double q1, q3, iqr;
    if (n == 1) { q1 = 0; q3 = a[0]; iqr = a[0]; }                    /* common.hpp:49-52 */
    else {
        const long half = n / 2;
        q1 = median_sorted(a, half);
        q3 = median_sorted(a + half + n % 2, n - (half + n % 2));
        iqr = q3 - q1;
    }
    const double low = q1 - 1.25 * iqr, high = q3 + 1.25 * iqr;       /* icp.cpp:104-105, IQR_TUCHEY common.hpp:15 */
    if (bounds2) { bounds2[0] = low; bounds2[1] = high; }
    long c = 0;
    for (long i = 0; i < n; ++i)
        if (d[i] >= low && d[i] <= high) { if (out) memcpy(out + 3 * c, xyz + 3 * i, 3 * sizeof(double)); ++c; }
    free(d); free(a);
    return c;
}

void lo_voxelize(const double *xyz, long n, double v, double *src, long *n_src, double *down, long *n_down) {
    const long nd = lo_voxel_downsample(xyz, n, v * 0.5, down, NULL);     /* icp.cpp:129 */
    double *s0 = (double *)malloc(sizeof(double) * 3 * (size_t)(nd > 0 ? nd : 1));
    const long ns0 = lo_voxel_downsample(down, nd, v * 1.5, s0, NULL);    /* :130 */
    *n_src = lo_iqr(s0, ns0, src, NULL);                                  /* :133 */
    *n_down = nd;
    free(s0);
}

/* ================================================================================================
 * Adaptive threshold: helpers/threshold.cpp
 * ============================================================================================== */
void lo_threshold_init(lo_threshold *a, double init_th, double min_motion, double max_range) {
    a->init_threshold = init_th; a->min_motion_th = min_motion; a->max_range = max_range;
    a->model_error_sq = 0.0; a->num_samples = 0;
    const double id[7] = {0, 0, 0, 1, 0, 0, 0};
    memcpy(a->dev, id, sizeof id);
}
/* theta = Eigen::AngleAxisd(model_dev.rotationMatrix()).angle(): quaternion -> matrix
 * (Eigen Quaternion::toRotationMatrix) -> quaternion (Eigen quaternionbase_assign_impl<.,3,3>)
 * -> 2*atan2(|vec|, |w|) (Eigen AngleAxis::operator=(Quaternion)). */
static double angle_of(const double *q) {
    const double x = q[0], y = q[1], z = q[2], w = q[3];
    const double tx = 2 * x, ty = 2 * y, tz = 2 * z;
    const double twx = tx * w, twy = ty * w, twz = tz * w, txx = tx * x, txy = ty * x, txz = tz * x, tyy = ty * y, tyz = tz * y, tzz = tz * z;
    double m[3][3];
    m[0][0] = 1 - (tyy + tzz); m[0][1] = txy - twz; m[0][2] = txz + twy;
    m[1][0] = txy + twz; m[1][1] = 1 - (txx + tzz); m[1][2] = tyz - twx;
    m[2][0] = txz - twy; m[2][1] = tyz + twx; m[2][2] = 1 - (txx + tyy);
    double c[4]; /* x y z w */
    double t = (m[0][0] + m[1][1]) + m[2][2];
    if (t > 0) {
        t = sqrt(t + 1.0);
        c[3] = 0.5 * t; t = 0.5 / t;
        c[0] = (m[2][1] - m[1][2]) * t; c[1] = (m[0][2] - m[2][0]) * t; c[2] = (m[1][0] - m[0][1]) * t;
    } else {
        int i = 0;
        if (m[1][1] > m[0][0]) i = 1;
        if (m[2][2] > m[i][i]) i = 2;
        const int j = (i + 1) % 3, k = (j + 1) % 3;
        t = sqrt(m[i][i] - m[j][j] - m[k][k] + 1.0);
        c[i] = 0.5 * t; t = 0.5 / t;
        c[3] = (m[k][j] - m[j][k]) * t; c[j] = (m[j][i] + m[i][j]) * t; c[k] = (m[k][i] + m[i][k]) * t;
    }
    const double n = sqrt(sqn3(c[0], c[1], c[2]));
    if (n != 0.0) return 2.0 * atan2(n, fabs(c[3]));
    return 0.0;
}
double lo_threshold_step(lo_threshold *a, const double *dev7) {
    memmove(a->dev, dev7, 7 * sizeof(double));
    const double theta = angle_of(a->dev);
    const double delta_rot = 2.0 * a->max_range * sin(theta / 2.0);
    const double delta_trans = sqrt(sqn3(a->dev[4], a->dev[5], a->dev[6]));
    const double model_error = delta_rot + delta_trans;               /* threshold.cpp:5-12 */
    if (model_error > a->min_motion_th) { a->model_error_sq += model_error * model_error; a->num_samples++; }
    if (a->num_samples < 1) return a->init_threshold;
    return sqrt(a->model_error_sq / a->num_samples);                  /* :16-28 */
}

/* ================================================================================================
 * KissICP: icp.cpp:36-86, :138-163
 * ============================================================================================== */
struct lo_kiss {
    double voxel_size, max_range, min_motion_th, initial_threshold, estimation_threshold;
    int cap, deskew, icp_max_iteration;
    lo_threshold th;
    lo_map *map;
    double *poses; long n_poses, poses_cap;
    int last_iters; double last_sigma;
};
lo_kiss *lo_kiss_create(double voxel_size, double max_range, int cap, int deskew, double min_motion_th,
                        int icp_max_iteration, double initial_threshold, double estimation_threshold) {
    lo_kiss *k = (lo_kiss *)calloc(1, sizeof(lo_kiss));
    k->voxel_size = voxel_size; k->max_range = max_range; k->cap = cap; k->deskew = deskew;
    k->min_motion_th = min_motion_th; k->icp_max_iteration = icp_max_iteration;
    k->initial_threshold = initial_threshold; k->estimation_threshold = estimation_threshold;
    lo_threshold_init(&k->th, initial_threshold, min_motion_th, max_range);   /* icp.hpp:35-39 */
    k->map = lo_map_create(voxel_size, max_range, cap);
    return k;
}
void lo_kiss_destroy(lo_kiss *k) { if (k) { lo_map_destroy(k->map); free(k->poses); free(k); } }
long lo_kiss_num_poses(const lo_kiss *k) { return k->n_poses; }
void lo_kiss_pose(const lo_kiss *k, long i, double *p) { memcpy(p, k->poses + 7 * i, 7 * sizeof(double)); }
lo_map *lo_kiss_map(lo_kiss *k) { return k->map; }
void lo_kiss_set_mode(lo_kiss *k, int icp_mode) { lo_map_set_mode(k->map, icp_mode); }
int lo_kiss_last_iterations(const lo_kiss *k) { return k->last_iters; }
double lo_kiss_last_sigma(const lo_kiss *k) { return k->last_sigma; }

static int kiss_has_moved(const lo_kiss *k) { /* icp.cpp:156-163 */
    if (k->n_poses == 0) return 0;
    double fi[7], d[7];
    lo_se3_inv(k->poses, fi);
    lo_se3_mul(fi, k->poses + 7 * (k->n_poses - 1), d);
    return sqrt(sqn3(d[4], d[5], d[6])) > 5.0 * k->min_motion_th;
}

void lo_kiss_register_points(lo_kiss *k, const double *xyz, long n, double *down, long *n_down, double *src,
                             long *n_src, double *pose7) { /* icp.cpp:58-86 */
    lo_voxelize(xyz, n, k->voxel_size, src, n_src, down, n_down);                 /* :61 */
    double sigma;                                                                 /* :66, :138-144 */
    if (!kiss_has_moved(k)) sigma = k->initial_threshold;
    else sigma = lo_threshold_step(&k->th, k->th.dev);
    const double id[7] = {0, 0, 0, 1, 0, 0, 0};
    double pred[7], last[7], init[7];
    memcpy(pred, id, sizeof id);
    if (k->n_poses >= 2) {                                                        /* :146-154 */
        double inv[7];
        lo_se3_inv(k->poses + 7 * (k->n_poses - 2), inv);
        lo_se3_mul(inv, k->poses + 7 * (k->n_poses - 1), pred);
    }
    if (k->n_poses == 0) memcpy(last, id, sizeof id); else memcpy(last, k->poses + 7 * (k->n_poses - 1), sizeof last);
    lo_se3_mul(last, pred, init);                                                 /* :69-71 */
    double newp[7];
    k->last_iters = lo_icp(k->map, src, *n_src, init, 3.0 * sigma, sigma / 3.0, k->icp_max_iteration,
                           k->estimation_threshold, newp, NULL, NULL, NULL, NULL); /* :74-76 */
    k->last_sigma = sigma;
    double ii[7], dev[7];
    lo_se3_inv(init, ii);
    lo_se3_mul(ii, newp, dev);                                                    /* :78 */
    memcpy(k->th.dev, dev, sizeof dev);                                           /* :79 */
    lo_map_update(k->map, down, *n_down, newp);                                   /* :81 */
    if (k->n_poses == k->poses_cap) {
        k->poses_cap = k->poses_cap ? 2 * k->poses_cap : 64;
        k->poses = (double *)realloc(k->poses, sizeof(double) * 7 * (size_t)k->poses_cap);
    }
    memcpy(k->poses + 7 * k->n_poses, newp, sizeof newp);                         /* :82 */
    ++k->n_poses;
    memcpy(pose7, newp, sizeof newp);
}

void lo_kiss_register_cloud(lo_kiss *k, const float *xyz, const double *ts, long n, double *down, long *n_down,
                            double *src, long *n_src, double *pose7) { /* icp.cpp:36-55 */
    double *frame = (double *)malloc(sizeof(double) * 3 * (size_t)(n > 0 ? n : 1));
    if (k->deskew && k->n_poses > 2)                                              /* :40-46 */
        lo_deskew(xyz, ts, n, k->poses + 7 * (k->n_poses - 2), k->poses + 7 * (k->n_poses - 1), frame);
    else
        for (long i = 0; i < 3 * n; ++i) frame[i] = (double)xyz[i];               /* pointcloud2eigen */
    lo_kiss_register_points(k, frame, n, down, n_down, src, n_src, pose7);
    free(frame);
}
