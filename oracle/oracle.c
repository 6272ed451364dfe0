/*
 * CPU oracle, compiled form: plain-C float64 restatement of the reference hot path.
 *
 * TEST INFRASTRUCTURE ONLY.  Built into oracle/_build/liboracle.so by oracle/Makefile and
 * loaded (ctypes) only by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg.
 * The product library never links, loads or calls it.
 *
 * Build with -ffp-contract=off: every product and sum below is rounded separately, as
 * CPython / NumPy scalar arithmetic does.
 *
 * Reference (paths relative to /root/reference, aliases as in SURVEY.md):
 *   [ICP]  W9_Fusion Localization (LiDAR Odometry)/course_agv_slam/scripts/icp.py
 *   [MAP]  W12_LiDAR SLAM/w12-mapping/course_agv_slam/scripts/mapping.py
 *   [BRES] W12_LiDAR SLAM/w12-mapping/course_agv_slam/scripts/bresenham.py
 *
 * Pinning: tests/test_oracle.py checks every function here against oracle/pyref.py (the
 * literal Python form), which in turn is checked against the executed reference classes
 * and the committed golden vectors (tests/golden/).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

/* ------------------------------------------------------------------ ICP pieces */

/* np.linalg.norm(src[i] - tar[j]) of [ICP]:102 for a 2-vector.  NumPy evaluates it as sqrt(x.dot(x)), and the dot of
 * two float64 values goes to the BLAS ddot, whose scalar tail loop (`dot += y[i] * x[i]`, OpenBLAS kernel/x86_64/ddot.c,
 * built with FMA contraction for every FMA3 target) computes fma(x1, x1, x0 * x0): ONE rounding for the first product,
 * one for the fused second step.  That is what the unmodified reference returns in this container (NumPy 2.3.5,
 * OpenBLAS 0.3.30) and what tests/golden/icp_ties.npz pins on 10^4 near-tie cases -- a plain dx*dx + dy*dy disagrees
 * with the reference on 86 of them.  NumPy pins no arithmetic and the reference pins no NumPy (SURVEY.md section 8c),
 * so this is "the reference as run here", on x86-64 with FMA3 (any host of a B200). */
static inline double ref_norm2(double dx, double dy)
{
    return sqrt(__builtin_fma(dy, dy, dx * dx));
}

/* [ICP]:90-114  nearest neighbour: strict '<' on the norm (square root INCLUDED: sqrt merges neighbouring doubles,
 * and the ties it creates go to the lowest j), ascending j. */
void orc_nearest(const double *src_xy, int n, const double *tar_xy, int m,
                 double *dist_out, int32_t *idx_out)
{
    for (int i = 0; i < n; ++i) {
        const double sx = src_xy[2 * i], sy = src_xy[2 * i + 1];
        double best = INFINITY;
        int32_t arg = 0;
        double keep = 0.0;
        for (int j = 0; j < m; ++j) {
            const double dx = sx - tar_xy[2 * j];
            const double dy = sy - tar_xy[2 * j + 1];
            const double d = ref_norm2(dx, dy);
            if (d < best) {
                best = d;
                arg = j;
                keep = d;
            }
        }
        dist_out[i] = keep;
        idx_out[i] = arg;
    }
}

/* NumPy reduces contiguous float64 arrays pairwise (blocks of 128, 8 accumulators);
 * a plain left-to-right sum differs from it only in the last bits and the parity
 * tolerance (1e-12 against the reference) absorbs that. */
static void centroid(const double *xy, const int32_t *pick, int n, double *cx, double *cy)
{
    double sx = 0.0, sy = 0.0;
    for (int i = 0; i < n; ++i) {
        const int k = pick ? pick[i] : i;
        sx += xy[2 * k];
        sy += xy[2 * k + 1];
    }
    *cx = sx / (double)n;
    *cy = sy / (double)n;
}

/* [ICP]:149-179 with the SVD replaced by the closed-form proper rotation
 * theta = atan2(W10 - W01, W00 + W11), W = sum (b - cb)(a - ca)^T.
 * a = src[i], b = tar[pick[i]] (pick == NULL: b = tar[i]).  T is row-major 3x3. */
void orc_rigid_fit(const double *src_xy, const double *tar_xy, const int32_t *pick, int n,
                   double *T)
{
    double cax, cay, cbx, cby;
    centroid(src_xy, NULL, n, &cax, &cay);
    centroid(tar_xy, pick, n, &cbx, &cby);
    double w00 = 0.0, w01 = 0.0, w10 = 0.0, w11 = 0.0;
    for (int i = 0; i < n; ++i) {
        const int k = pick ? pick[i] : i;
        const double ax = src_xy[2 * i] - cax, ay = src_xy[2 * i + 1] - cay;
        const double bx = tar_xy[2 * k] - cbx, by = tar_xy[2 * k + 1] - cby;
        w00 += bx * ax;
        w01 += bx * ay;
        w10 += by * ax;
        w11 += by * ay;
    }
    const double cc = w00 + w11, ss = w10 - w01;
    const double h = hypot(cc, ss);
    double c = 1.0, s = 0.0;
    if (h > 0.0) {
        c = cc / h;
        s = ss / h;
    }
    T[0] = c;  T[1] = -s; T[2] = cbx - (c * cax - s * cay);
    T[3] = s;  T[4] = c;  T[5] = cby - (s * cax + c * cay);
    T[6] = 0.0; T[7] = 0.0; T[8] = 1.0;
}

/* [ICP]:38-88  one scan pair.  src_xy [n][2], tar_xy [m][2]; scratch sized by caller. */
/* *err_out: mean_error of the last iteration that ran ([ICP]:75), 0 when none did. */
static int icp_one(const double *tar_xy, int m, const double *src_xy, int n, int max_iter,
                   double tol, double *T_out, double *err_out, double *cur, double *dist, int32_t *idx)
{
    memcpy(cur, src_xy, sizeof(double) * 2 * (size_t)n);
    double prev = 0.0, err = 0.0;
    int iters = 0;
    double T[9];
    for (int it = 0; it < max_iter; ++it) {
        orc_nearest(cur, n, tar_xy, m, dist, idx);
        orc_rigid_fit(cur, tar_xy, idx, n, T);
        for (int i = 0; i < n; ++i) { /* [ICP]:71  src = T . src (row . column, left to right) */
            const double x = cur[2 * i], y = cur[2 * i + 1];
            cur[2 * i] = T[0] * x + T[1] * y + T[2];
            cur[2 * i + 1] = T[3] * x + T[4] * y + T[5];
        }
        ++iters;
        double total = 0.0;
        for (int i = 0; i < n; ++i) total += dist[i];
        err = total / (double)n;               /* [ICP]:75 distances from BEFORE the move */
        if (fabs(prev - err) < tol) break;     /* [ICP]:76 strict '<' */
        prev = err;
    }
    orc_rigid_fit(src_xy, cur, NULL, n, T_out); /* [ICP]:81 final re-fit */
    *err_out = err;
    return iters;
}

/* Batch of independent pairs.  tar [P][m][2], src [P][n][2] float64; T_out [P][9]; err_out [P] (may be NULL) the
 * mean_error of each pair's last iteration, summed left to right. */
int orc_icp_batch_err(const double *tar_xy, const double *src_xy, int pairs, int n, int m,
                      int max_iter, double tol, double *T_out, int32_t *iters_out, double *err_out)
{
    if (pairs < 0 || n <= 0 || m <= 0 || max_iter < 0) return -1;
    {
        double *cur = (double *)malloc(sizeof(double) * 2 * (size_t)n);
        double *dist = (double *)malloc(sizeof(double) * (size_t)n);
        int32_t *idx = (int32_t *)malloc(sizeof(int32_t) * (size_t)n);
        for (int p = 0; p < pairs; ++p) {
            double err;
            iters_out[p] = icp_one(tar_xy + (size_t)p * m * 2, m, src_xy + (size_t)p * n * 2, n,
                                   max_iter, tol, T_out + (size_t)p * 9, &err, cur, dist, idx);
            if (err_out) err_out[p] = err;
        }
        free(cur);
        free(dist);
        free(idx);
    }
    return 0;
}

int orc_icp_batch(const double *tar_xy, const double *src_xy, int pairs, int n, int m,
                  int max_iter, double tol, double *T_out, int32_t *iters_out)
{
    return orc_icp_batch_err(tar_xy, src_xy, pairs, n, m, max_iter, tol, T_out, iters_out, NULL);
}

/* ------------------------------------------------------------------ Bresenham / grid */

/* [BRES]:2-58.  Writes up to cap (x,y) pairs into out_xy, returns the path length
 * (max(|dx|,|dy|)+1, or 0 for a same-cell segment) even when it exceeds cap. */
int64_t orc_bresenham(int64_t x0, int64_t y0, int64_t x1, int64_t y1, int32_t *out_xy,
                      int64_t cap)
{
    if (x0 == x1 && y0 == y1) return 0;
    const int steep = llabs(y1 - y0) > llabs(x1 - x0);
    if (steep) {
        int64_t t = x0; x0 = y0; y0 = t;
        t = x1; x1 = y1; y1 = t;
    }
    const int flipped = x0 > x1;
    if (flipped) {
        int64_t t = x0; x0 = x1; x1 = t;
        t = y0; y0 = y1; y1 = t;
    }
    const int64_t span = x1 - x0;
    const int64_t rise = llabs(y1 - y0);
    const double slope = (double)rise / (double)span;
    double acc = 0.0;
    int64_t minor = y0;
    const int64_t inc = (y0 < y1) ? 1 : -1;
    const int64_t len = span + 1;
    for (int64_t k = 0; k < len; ++k) {
        const int64_t major = x0 + k;
        const int64_t slot = flipped ? (len - 1 - k) : k;
        if (slot < cap) {
            out_xy[2 * slot] = (int32_t)(steep ? minor : major);
            out_xy[2 * slot + 1] = (int32_t)(steep ? major : minor);
        }
        acc += slope;
        if (acc >= 0.5) {
            minor += inc;
            acc -= 1.0;
        }
    }
    return len;
}

/* [MAP]:33-36  int(S * (v + H)): float64, truncation toward zero. */
static inline int64_t to_cell(double v, double cells_per_m, double off)
{
    return (int64_t)(cells_per_m * (v + off));
}

/* One beam of [MAP]:29-50 in integer form; endpoints and sensor position in float64 world coordinates.
 * Returns 0, or -1 on a coordinate the reference would raise on (NaN anywhere, inf in fy / centre). */
static int raycast_beam(int32_t *hit, int32_t *miss, int xw, int yw, double cells_per_m, double off_x,
                        double off_y, double fx, double fy, double fcx, double fcy, int64_t *visits)
{
    if (isinf(fx)) return 0;                                   /* [MAP]:30 */
    if (isnan(fx) || !isfinite(fy) || !isfinite(fcx) || !isfinite(fcy)) return -1;
    int64_t x0 = to_cell(fcx, cells_per_m, off_x), y0 = to_cell(fcy, cells_per_m, off_y);
    int64_t x1 = to_cell(fx, cells_per_m, off_x), y1 = to_cell(fy, cells_per_m, off_y);
    if (x0 == x1 && y0 == y1) return 0;
    const int steep = llabs(y1 - y0) > llabs(x1 - x0);
    if (steep) {
        int64_t t = x0; x0 = y0; y0 = t;
        t = x1; x1 = y1; y1 = t;
    }
    const int flipped = x0 > x1;
    if (flipped) {
        int64_t t = x0; x0 = x1; x1 = t;
        t = y0; y0 = y1; y1 = t;
    }
    const int64_t span = x1 - x0;
    const double slope = (double)llabs(y1 - y0) / (double)span;
    const int64_t inc = (y0 < y1) ? 1 : -1;
    /* the endpoint (obstacle) is the last canonical cell unless the trace was flipped */
    const int64_t hit_k = flipped ? 0 : span;
    double acc = 0.0;
    int64_t minor = y0;
    for (int64_t k = 0; k <= span; ++k) {
        const int64_t major = x0 + k;
        const int64_t px = steep ? minor : major;
        const int64_t py = steep ? major : minor;
        if (px >= 0 && px < xw && py >= 0 && py < yw) {
            const size_t cell = (size_t)px * (size_t)yw + (size_t)py;
            if (k == hit_k) hit[cell] += 1; else miss[cell] += 1;
            ++*visits;
        }
        acc += slope;
        if (acc >= 0.5) {
            minor += inc;
            acc -= 1.0;
        }
    }
    return 0;
}

/* [MAP]:22-51 in integer form: K scans x N beams into hit/miss [xw][yw] (x-major), float32 endpoints.
 * Returns in-grid cell visits, or -1 on a non-finite coordinate the reference would raise on. */
int64_t orc_grid_raycast(int32_t *hit, int32_t *miss, int xw, int yw, double cells_per_m,
                         double off_x, double off_y, const float *ox, const float *oy,
                         const float *cx, const float *cy, int scans, int beams)
{
    int64_t visits = 0;
    for (int s = 0; s < scans; ++s) {
        const double fcx = (double)cx[s], fcy = (double)cy[s];
        if (!isfinite(fcx) || !isfinite(fcy)) return -1;
        for (int b = 0; b < beams; ++b)
            if (raycast_beam(hit, miss, xw, yw, cells_per_m, off_x, off_y, (double)ox[(size_t)s * beams + b],
                             (double)oy[(size_t)s * beams + b], fcx, fcy, &visits))
                return -1;
    }
    return visits;
}

/* The same on float64 endpoints / sensor positions: the dtype [MAP]:22-51 is called with by slam_ekf.py:89-90
 * (obs and xEst are float64), so int(10*(v+10)) sees the unrounded value. */
int64_t orc_grid_raycast_f64(int32_t *hit, int32_t *miss, int xw, int yw, double cells_per_m,
                             double off_x, double off_y, const double *ox, const double *oy,
                             const double *cx, const double *cy, int scans, int beams)
{
    int64_t visits = 0;
    for (int s = 0; s < scans; ++s) {
        const double fcx = cx[s], fcy = cy[s];
        for (int b = 0; b < beams; ++b)
            if (raycast_beam(hit, miss, xw, yw, cells_per_m, off_x, off_y, ox[(size_t)s * beams + b],
                             oy[(size_t)s * beams + b], fcx, fcy, &visits))
                return -1;
    }
    return visits;
}

/* Raw scans: laserToNumpy (slam_ekf.py:115-123) + u2T(xEst).dot(np_msg) (slam_ekf.py:130-137,89) + the update,
 * per beam in float64, products and sums rounded separately, left to right.  pose4 [scans][4] = x, y,
 * cos(yaw), sin(yaw); beam_cs [beams][2] = cos, sin of the beam angle; clamp > 0 replaces +inf ranges. */
int64_t orc_grid_raycast_ranges(int32_t *hit, int32_t *miss, int xw, int yw, double cells_per_m,
                                double off_x, double off_y, const float *ranges, const double *pose4,
                                const double *beam_cs, double clamp, int scans, int beams)
{
    int64_t visits = 0;
    for (int s = 0; s < scans; ++s) {
        const double x = pose4[4 * s], y = pose4[4 * s + 1], cw = pose4[4 * s + 2], sw = pose4[4 * s + 3];
        for (int b = 0; b < beams; ++b) {
            double r = (double)ranges[(size_t)s * beams + b];
            if (clamp > 0.0 && r == INFINITY) r = clamp;
            const double px = beam_cs[2 * b] * r, py = beam_cs[2 * b + 1] * r;
            const double fx = (cw * px + (-sw) * py) + x;
            const double fy = (sw * px + cw * py) + y;
            if (raycast_beam(hit, miss, xw, yw, cells_per_m, off_x, off_y, fx, fy, x, y, &visits)) return -1;
        }
    }
    return visits;
}

/* SURVEY.md section 8a row A6: counts -> score (float64) and occupancy {0, 50, 100}. */
void orc_grid_finalize(const int32_t *hit, const int32_t *miss, int64_t cells, double w_hit,
                       double w_miss, double thresh, double *score, int8_t *pmap)
{
    for (int64_t i = 0; i < cells; ++i) {
        const double v = w_miss * (double)miss[i] + w_hit * (double)hit[i];
        if (score) score[i] = v;
        if (pmap) pmap[i] = (hit[i] == 0 && miss[i] == 0) ? 50 : (v > thresh ? 100 : 0);
    }
}
