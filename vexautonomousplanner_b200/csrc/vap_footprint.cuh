// vap_footprint.cuh -- does the robot's rectangle stay on the field and clear the keep-out boxes along every row of a
// trajectory export ({0, t, x_in, y_in, heading, v, omega}, vap_export_rows or the rows read back from a saved .txt)?
//
// Geometry per row (x, y, heading h as written; h is CCW from +x in the export frame, turn rows carry absolute
// headings, and a reversed segment's h - pi leaves the centred rectangle unchanged): the corners are
// (x + a cos h - b sin h, y + a sin h + b cos h) for a = +-hl, b = +-hw.
//   wall margin  max over the corners of max(xmin - cx, cx - xmax, ymin - cy, cy - ymax); negative = clearance.
//   box distance signed: with overlap on all four separating axes (the box's x and y, the robot's heading and its
//                normal) minus the smallest overlap (the penetration depth), else the Euclidean distance between
//                the two rectangles.  The vertex-edge minimum of two disjoint convex polygons equals the smaller of
//                "robot corner to box" (axis-aligned clamp) and "box corner to robot" (clamp in the robot's frame),
//                which is what is evaluated here.
//   violation    wall margin > tol, some box distance < -tol, or x, y or h not finite (kind 1; no geometry).
// One CTA per path; every per-path result is a selection (min / max with the lowest row, then the lowest box, winning
// ties) or an integer count, so it does not depend on the launch shape and is bit-identical run to run.
#pragma once

#define FP_MAX_BOXES 64
#define FP_ROWS 0             // out_i64 columns
#define FP_FIRST_ROW 1        // first violating row, -1 none
#define FP_FIRST_KIND 2       // -1 none, 0 wall, 1 non-finite, 2 + k keep-out box k
#define FP_VIOLATING 3        // rows that violate
#define FP_WORST_WALL_ROW 4   // row of the largest wall margin (-1 without a finite row)
#define FP_NEAREST_ROW 5      // row of the smallest box distance (-1 when K = 0 or without a finite row)
#define FP_NEAREST_BOX 6      // that box (-1 likewise)
#define FP_NI 7
#define FP_FIRST_T 0          // out_f64 columns: t of the first violation (NaN none)
#define FP_WORST_WALL 1       // largest wall margin (-inf without a finite row)
#define FP_WORST_WALL_T 2
#define FP_NEAREST 3          // smallest box distance (+inf when K = 0 or without a finite row)
#define FP_NEAREST_T 4
#define FP_MAX_STEP 5         // largest corner displacement between consecutive finite rows (0 with fewer than two)
#define FP_NF 6
#define FP_THREADS 256

struct FpArgs {               // passed by value: validated on the host, copied to shared memory by every CTA
    double hl, hw, xmin, xmax, ymin, ymax, tol;
    int K;
    double box[FP_MAX_BOXES][4];    // {x0, y0, x1, y1}
};

struct FpAcc {
    long long first, count, worst_r, near_r;
    double worst, near, step;
    int first_kind, near_k;
};

#define FP_NONE 0x7fffffffffffffffLL

__device__ __forceinline__ void fp_merge(FpAcc& a, const FpAcc& o)
{
    if (o.first < a.first) { a.first = o.first; a.first_kind = o.first_kind; }
    a.count += o.count;
    if (o.worst > a.worst || (o.worst == a.worst && o.worst_r < a.worst_r)) { a.worst = o.worst; a.worst_r = o.worst_r; }
    if (o.near < a.near || (o.near == a.near && (o.near_r < a.near_r || (o.near_r == a.near_r && o.near_k < a.near_k)))) {
        a.near = o.near; a.near_r = o.near_r; a.near_k = o.near_k;
    }
    a.step = fmax(a.step, o.step);
}

__device__ __forceinline__ FpAcc fp_shfl(const FpAcc& a, int o)
{
    FpAcc r;
    r.first = __shfl_xor_sync(0xffffffffu, a.first, o);
    r.count = __shfl_xor_sync(0xffffffffu, a.count, o);
    r.worst_r = __shfl_xor_sync(0xffffffffu, a.worst_r, o);
    r.near_r = __shfl_xor_sync(0xffffffffu, a.near_r, o);
    r.worst = __shfl_xor_sync(0xffffffffu, a.worst, o);
    r.near = __shfl_xor_sync(0xffffffffu, a.near, o);
    r.step = __shfl_xor_sync(0xffffffffu, a.step, o);
    r.first_kind = __shfl_xor_sync(0xffffffffu, a.first_kind, o);
    r.near_k = __shfl_xor_sync(0xffffffffu, a.near_k, o);
    return r;
}

__device__ __forceinline__ bool fp_finite(const double* row)
{
    return isfinite(row[2]) && isfinite(row[3]) && isfinite(row[4]);
}

__device__ __forceinline__ void fp_corners(const double* row, double hl, double hw, double* cx, double* cy, double& c, double& s)
{
    const double x = row[2], y = row[3];
    sincos(row[4], &s, &c);
    const double ac = hl * c, as = hl * s, bc = hw * c, bs = hw * s;
    cx[0] = x + ac - bs; cy[0] = y + as + bc;         // (a, b) = (+hl, +hw)
    cx[1] = x + ac + bs; cy[1] = y + as - bc;         // (+hl, -hw)
    cx[2] = x - ac - bs; cy[2] = y - as + bc;         // (-hl, +hw)
    cx[3] = x - ac + bs; cy[3] = y - as - bc;         // (-hl, -hw)
}

// bx[k] = {x0, y0, x1, y1, centre x, centre y, half width, half height}
__global__ void __launch_bounds__(FP_THREADS) k_footprint_check(long long B, const double* __restrict__ rows,
                                                                const long long* __restrict__ row_off, const FpArgs a,
                                                                long long* __restrict__ out_i, double* __restrict__ out_f)
{
    __shared__ double bx[FP_MAX_BOXES][8];
    __shared__ FpAcc part[FP_THREADS / 32];
    const int K = a.K;
    for (int k = threadIdx.x; k < K; k += blockDim.x) {
        const double x0 = a.box[k][0], y0 = a.box[k][1], x1 = a.box[k][2], y1 = a.box[k][3];
        bx[k][0] = x0; bx[k][1] = y0; bx[k][2] = x1; bx[k][3] = y1;
        bx[k][4] = 0.5 * (x0 + x1); bx[k][5] = 0.5 * (y0 + y1); bx[k][6] = 0.5 * (x1 - x0); bx[k][7] = 0.5 * (y1 - y0);
    }
    __syncthreads();
    const double hl = a.hl, hw = a.hw, tol = a.tol;
    const double inf = __longlong_as_double(0x7ff0000000000000LL);
    for (long long b = blockIdx.x; b < B; b += gridDim.x) {
        const long long r0 = row_off[b], n = row_off[b + 1] - r0;
        FpAcc acc = {FP_NONE, 0, FP_NONE, FP_NONE, -inf, inf, 0.0, -1, -1};
        for (long long r = threadIdx.x; r < n; r += blockDim.x) {
            const double* row = rows + (size_t)(r0 + r) * 7;
            if (!fp_finite(row)) {
                if (acc.first == FP_NONE) { acc.first = r; acc.first_kind = 1; }
                acc.count++;
                continue;
            }
            double cx[4], cy[4], c, s;
            fp_corners(row, hl, hw, cx, cy, c, s);
            double m = -inf, rxmin = cx[0], rxmax = cx[0], rymin = cy[0], rymax = cy[0];
#pragma unroll
            for (int i = 0; i < 4; i++) {
                m = fmax(m, fmax(fmax(a.xmin - cx[i], cx[i] - a.xmax), fmax(a.ymin - cy[i], cy[i] - a.ymax)));
                rxmin = fmin(rxmin, cx[i]); rxmax = fmax(rxmax, cx[i]);
                rymin = fmin(rymin, cy[i]); rymax = fmax(rymax, cy[i]);
            }
            if (m > acc.worst) { acc.worst = m; acc.worst_r = r; }
            if (r > 0 && fp_finite(row - 7)) {
                double px[4], py[4], pc, ps;
                fp_corners(row - 7, hl, hw, px, py, pc, ps);
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    const double dx = cx[i] - px[i], dy = cy[i] - py[i];
                    acc.step = fmax(acc.step, sqrt(dx * dx + dy * dy));
                }
            }
            const double x = row[2], y = row[3];
            const double pu = x * c + y * s, pv = y * c - x * s;        // the centre on the heading and on its normal
            const double ac_ = fabs(c), as_ = fabs(s);
            double dmin = inf;
            int kmin = -1, kviol = -1;
            for (int k = 0; k < K; k++) {
                const double* q = bx[k];
                const double ox = fmin(rxmax, q[2]) - fmax(rxmin, q[0]);
                const double oy = fmin(rymax, q[3]) - fmax(rymin, q[1]);
                const double bu = q[4] * c + q[5] * s, bv = q[5] * c - q[4] * s;
                const double eu = q[6] * ac_ + q[7] * as_, ev = q[6] * as_ + q[7] * ac_;
                const double ou = fmin(pu + hl, bu + eu) - fmax(pu - hl, bu - eu);
                const double ov = fmin(pv + hw, bv + ev) - fmax(pv - hw, bv - ev);
                double d;
                if (ox > 0 && oy > 0 && ou > 0 && ov > 0) {
                    d = -fmin(fmin(ox, oy), fmin(ou, ov));
                } else {
                    double d2 = inf;
#pragma unroll
                    for (int i = 0; i < 4; i++) {                       // robot corner -> box
                        const double ex = fmax(fmax(q[0] - cx[i], cx[i] - q[2]), 0.0);
                        const double ey = fmax(fmax(q[1] - cy[i], cy[i] - q[3]), 0.0);
                        d2 = fmin(d2, ex * ex + ey * ey);
                    }
#pragma unroll
                    for (int j = 0; j < 4; j++) {                       // box corner -> robot, in the robot's frame
                        const double wx = (j & 1) ? q[2] : q[0], wy = (j & 2) ? q[3] : q[1];
                        const double eu2 = fmax(fabs(wx * c + wy * s - pu) - hl, 0.0);
                        const double ev2 = fmax(fabs(wy * c - wx * s - pv) - hw, 0.0);
                        d2 = fmin(d2, eu2 * eu2 + ev2 * ev2);
                    }
                    d = sqrt(d2);
                }
                if (d < dmin) { dmin = d; kmin = k; }
                if (kviol < 0 && d < -tol) kviol = k;
            }
            if (kmin >= 0 && dmin < acc.near) { acc.near = dmin; acc.near_r = r; acc.near_k = kmin; }
            const int kind = m > tol ? 0 : (kviol >= 0 ? 2 + kviol : -1);
            if (kind >= 0) {
                if (acc.first == FP_NONE) { acc.first = r; acc.first_kind = kind; }
                acc.count++;
            }
        }
        for (int o = 16; o > 0; o >>= 1) fp_merge(acc, fp_shfl(acc, o));
        const int warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
        if ((threadIdx.x & 31) == 0) part[warp] = acc;
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < nw; w++) fp_merge(acc, part[w]);
            const double qnan = __longlong_as_double(0x7ff8000000000000LL);
            long long* oi = out_i + (size_t)b * FP_NI;
            double* of = out_f + (size_t)b * FP_NF;
            const bool hit = acc.first != FP_NONE, fin = acc.worst_r != FP_NONE, near = acc.near_r != FP_NONE;
            oi[FP_ROWS] = n;
            oi[FP_FIRST_ROW] = hit ? acc.first : -1;
            oi[FP_FIRST_KIND] = hit ? acc.first_kind : -1;
            oi[FP_VIOLATING] = acc.count;
            oi[FP_WORST_WALL_ROW] = fin ? acc.worst_r : -1;
            oi[FP_NEAREST_ROW] = near ? acc.near_r : -1;
            oi[FP_NEAREST_BOX] = near ? acc.near_k : -1;
            of[FP_FIRST_T] = hit ? rows[(size_t)(r0 + acc.first) * 7 + 1] : qnan;
            of[FP_WORST_WALL] = acc.worst;
            of[FP_WORST_WALL_T] = fin ? rows[(size_t)(r0 + acc.worst_r) * 7 + 1] : qnan;
            of[FP_NEAREST] = acc.near;
            of[FP_NEAREST_T] = near ? rows[(size_t)(r0 + acc.near_r) * 7 + 1] : qnan;
            of[FP_MAX_STEP] = acc.step;
        }
        __syncthreads();                                               // part[] is reused by the next path
    }
}
