// vap_pairs.cuh -- two robots running their routes at the same time: where do their rectangles first touch?
//
// Input: two row sets of export rows ({0, t, x_in, y_in, heading, v, omega}, vap_export_rows or rows read back from
// saved .txt files), turned once into pose planes {t, x, y, cos h, sin h} (k_pose_planes), and a list of pairs
// (route a of set A, route b of set B).  Robot A is a rectangle centred on (x, y), hl_a along its heading and hw_a
// across it; robot B likewise with its own hl_b, hw_b.  Both start at t = 0 of their own rows.
//
//   events       every row of either route is one event (na + nb per pair).  At the event of A's row i, A is at row
//                i and B at its held pose: its last row with t <= t_i (upper_bound - 1 on B's t plane), clamped to
//                B's first row before it starts; after its last row B stays parked there.  B's rows likewise.
//   distance     signed: when the rectangles overlap on all four separating axes (each robot's heading and normal)
//                minus the smallest overlap (the penetration depth), else the Euclidean distance, evaluated as the
//                smaller of "A's corners clamped into B's frame" and "B's corners clamped into A's frame" (the
//                vertex-edge minimum of two disjoint convex polygons).  pc_signed_distance is symmetric bit for bit:
//                swapping the robots swaps two calls whose results are combined by min.
//   contact      distance < min_gap.
//   order        events are keyed (t, side, row), side A = 0 before B = 1.  The first contact is the contact with the
//                smallest key; the nearest event the smallest distance, the smallest key winning ties.  Every per-pair
//                result is such a selection, a max or an integer count, so it does not depend on the launch shape.
//   step         the largest corner move of either robot between consecutive rows of its own route: between two
//                consecutive events only one robot moves, by one such step, so it is the check's resolution.
//   invalid      a route without rows, with a non-finite t, x, y or heading, or whose t decreases is not checked
//                (k_pose_planes records the first such row and why).  Coordinates are inches on a field: beyond about
//                1e307 their differences overflow and the distance means nothing, though it is never NaN (fmin / fmax
//                drop NaN operands), so a checked pair always has a nearest event.
#pragma once

#define PC_BAD_NONE 0         // bad[b] = {first invalid row (-1 none or no rows), reason}
#define PC_BAD_EMPTY 1        // no rows
#define PC_BAD_NONFINITE 2    // t, x, y or heading not finite at that row
#define PC_BAD_DECREASING 3   // t at that row is smaller than at the row before
#define PC_OK 0               // out_i64 status
#define PC_A_INVALID 1
#define PC_B_INVALID 2
#define PC_BAD_INDEX 3        // a pair index outside 0 .. B - 1
#define PC_STATUS 0           // out_i64 columns
#define PC_EVENTS 1
#define PC_FIRST_SIDE 2       // -1 none
#define PC_FIRST_ROW 3
#define PC_CONTACTS 4
#define PC_NEAR_SIDE 5
#define PC_NEAR_ROW 6
#define PC_NI 7
#define PC_FIRST_T 0          // out_f64 columns: t of the first contact (NaN none)
#define PC_NEAR 1             // smallest distance (+inf when not checked)
#define PC_NEAR_T 2
#define PC_LAST_T_A 3         // NaN when not checked
#define PC_LAST_T_B 4
#define PC_MAX_STEP 5         // largest corner move between consecutive rows of either route
#define PC_NF 6
#define PC_THREADS 256

// ---- pose planes: planes[0..4][R] = t, x, y, cos h, sin h; bad[b] = {row, reason} ---------------------------------
__global__ void __launch_bounds__(PC_THREADS) k_pose_planes(long long B, const double* __restrict__ rows,
                                                            const long long* __restrict__ row_off, long long R,
                                                            double* __restrict__ planes, long long* __restrict__ bad)
{
    __shared__ unsigned long long first;           // 4 * row + reason of the first invalid row
    for (long long b = blockIdx.x; b < B; b += gridDim.x) {
        const long long r0 = row_off[b], n = row_off[b + 1] - r0;
        if (threadIdx.x == 0) first = ~0ull;
        __syncthreads();
        for (long long r = threadIdx.x; r < n; r += blockDim.x) {
            const double* row = rows + (size_t)(r0 + r) * 7;
            const double t = row[1], x = row[2], y = row[3], h = row[4];
            double s, c;
            sincos(h, &s, &c);
            const size_t k = (size_t)(r0 + r);
            planes[k] = t; planes[R + k] = x; planes[2 * R + k] = y; planes[3 * R + k] = c; planes[4 * R + k] = s;
            int why = 0;
            if (!isfinite(t) || !isfinite(x) || !isfinite(y) || !isfinite(h)) why = PC_BAD_NONFINITE;
            else if (r > 0 && t < (row - 7)[1]) why = PC_BAD_DECREASING;
            if (why) atomicMin(&first, 4ull * (unsigned long long)r + why);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            long long* o = bad + 2 * b;
            if (n == 0) { o[0] = -1; o[1] = PC_BAD_EMPTY; }
            else if (first == ~0ull) { o[0] = -1; o[1] = PC_BAD_NONE; }
            else { o[0] = (long long)(first >> 2); o[1] = (long long)(first & 3); }
        }
        __syncthreads();                                               // first is reset for the next route
    }
}

// ---- one robot's pose on its planes ----------------------------------------------------------------------------
struct PcPose {
    double x, y, c, s, hl, hw;
};

__device__ __forceinline__ PcPose pc_pose(const double* __restrict__ p, long long R, long long k, double hl, double hw)
{
    return PcPose{p[R + k], p[2 * R + k], p[3 * R + k], p[4 * R + k], hl, hw};
}

// Q's frame: the two SAT overlaps on Q's heading and normal, and the smallest squared distance of P's corners
// clamped into Q's rectangle.
__device__ __forceinline__ void pc_one_way(const PcPose& P, const PcPose& Q, double& ou, double& ov, double& d2)
{
    const double dx = P.x - Q.x, dy = P.y - Q.y;
    const double u = dx * Q.c + dy * Q.s, v = dy * Q.c - dx * Q.s;     // P's centre in Q's frame
    const double cd = P.c * Q.c + P.s * Q.s, sd = P.s * Q.c - P.c * Q.s;   // P's heading in Q's frame
    const double acd = fabs(cd), asd = fabs(sd);
    const double au = fabs(u), av = fabs(v);
    const double eu = P.hl * acd + P.hw * asd, ev = P.hl * asd + P.hw * acd;   // P's half-extents on Q's axes
    ou = fmin(Q.hl, au + eu) - fmax(-Q.hl, au - eu);                    // intersection of the two intervals
    ov = fmin(Q.hw, av + ev) - fmax(-Q.hw, av - ev);
    const double ac = P.hl * cd, as = P.hl * sd, bc = P.hw * cd, bs = P.hw * sd;
    d2 = __longlong_as_double(0x7ff0000000000000LL);
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const double a = (i & 1) ? -1.0 : 1.0, bsg = (i & 2) ? -1.0 : 1.0;
        const double cu = u + a * ac - bsg * bs, cv = v + a * as + bsg * bc;
        const double eu = fmax(fabs(cu) - Q.hl, 0.0), ev = fmax(fabs(cv) - Q.hw, 0.0);
        d2 = fmin(d2, eu * eu + ev * ev);
    }
}

__device__ __forceinline__ double pc_signed_distance(const PcPose& A, const PcPose& B)
{
    double oua, ova, d2a, oub, ovb, d2b;
    pc_one_way(B, A, oua, ova, d2a);       // on A's axes, B's corners into A
    pc_one_way(A, B, oub, ovb, d2b);       // on B's axes, A's corners into B
    if (oua > 0 && ova > 0 && oub > 0 && ovb > 0) return -fmin(fmin(oua, ova), fmin(oub, ovb));
    return sqrt(fmin(d2a, d2b));
}

// largest move of a corner between rows k - 1 and k of one route (sqrt is correctly rounded and monotone, so one sqrt
// of the largest square equals the largest of four)
__device__ __forceinline__ double pc_corner_step(const PcPose& p, const PcPose& q)
{
    double m2 = 0.0;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const double a = (i & 1) ? -p.hl : p.hl, b = (i & 2) ? -p.hw : p.hw;
        const double dx = (p.x + a * p.c - b * p.s) - (q.x + a * q.c - b * q.s);
        const double dy = (p.y + a * p.s + b * p.c) - (q.y + a * q.s + b * q.c);
        m2 = fmax(m2, dx * dx + dy * dy);
    }
    return sqrt(m2);
}

// last index k in [0, n) with t[k] <= key, 0 when there is none
__device__ __forceinline__ long long pc_held(const double* __restrict__ t, long long n, double key)
{
    long long lo = 0, hi = n;
    while (lo < hi) {
        const long long mid = (lo + hi) >> 1;
        if (t[mid] <= key) lo = mid + 1; else hi = mid;
    }
    return lo > 0 ? lo - 1 : 0;
}

struct PcAcc {
    double first_t, near, near_t, step;
    long long first_k, near_k, count;      // keys: side << 62 | row
};

#define PC_NONE 0x7fffffffffffffffLL

__device__ __forceinline__ bool pc_key_less(double t, long long k, double t2, long long k2)
{
    return t < t2 || (t == t2 && k < k2);
}

__device__ __forceinline__ void pc_merge(PcAcc& a, const PcAcc& o)
{
    if (pc_key_less(o.first_t, o.first_k, a.first_t, a.first_k)) { a.first_t = o.first_t; a.first_k = o.first_k; }
    if (o.near < a.near || (o.near == a.near && pc_key_less(o.near_t, o.near_k, a.near_t, a.near_k))) {
        a.near = o.near; a.near_t = o.near_t; a.near_k = o.near_k;
    }
    a.count += o.count;
    a.step = fmax(a.step, o.step);
}

__device__ __forceinline__ PcAcc pc_shfl(const PcAcc& a, int o)
{
    PcAcc r;
    r.first_t = __shfl_xor_sync(0xffffffffu, a.first_t, o);
    r.near = __shfl_xor_sync(0xffffffffu, a.near, o);
    r.near_t = __shfl_xor_sync(0xffffffffu, a.near_t, o);
    r.step = __shfl_xor_sync(0xffffffffu, a.step, o);
    r.first_k = __shfl_xor_sync(0xffffffffu, a.first_k, o);
    r.near_k = __shfl_xor_sync(0xffffffffu, a.near_k, o);
    r.count = __shfl_xor_sync(0xffffffffu, a.count, o);
    return r;
}

struct PcSide {               // one row set: planes[5][R], route b owns rows off[b] .. off[b+1]
    const double* planes;
    const long long* off;
    const long long* bad;
    long long B, R;
    double hl, hw;
};

// One CTA per pair; threads stride over the na + nb events.
__global__ void __launch_bounds__(PC_THREADS) k_pair_check(long long P, const long long* __restrict__ pairs, const PcSide sa,
                                                           const PcSide sb, double min_gap, long long* __restrict__ out_i,
                                                           double* __restrict__ out_f)
{
    __shared__ PcAcc part[PC_THREADS / 32];
    const double inf = __longlong_as_double(0x7ff0000000000000LL);
    const double qnan = __longlong_as_double(0x7ff8000000000000LL);
    for (long long p = blockIdx.x; p < P; p += gridDim.x) {
        const long long ia = pairs[2 * p], ib = pairs[2 * p + 1];
        long long* oi = out_i + (size_t)p * PC_NI;
        double* of = out_f + (size_t)p * PC_NF;
        const int status = (ia < 0 || ia >= sa.B || ib < 0 || ib >= sb.B) ? PC_BAD_INDEX
                         : sa.bad[2 * ia + 1] != PC_BAD_NONE ? PC_A_INVALID
                         : sb.bad[2 * ib + 1] != PC_BAD_NONE ? PC_B_INVALID : PC_OK;
        if (status != PC_OK) {                                         // uniform over the CTA
            if (threadIdx.x == 0) {
                oi[PC_STATUS] = status; oi[PC_EVENTS] = 0; oi[PC_FIRST_SIDE] = -1; oi[PC_FIRST_ROW] = -1;
                oi[PC_CONTACTS] = 0; oi[PC_NEAR_SIDE] = -1; oi[PC_NEAR_ROW] = -1;
                of[PC_FIRST_T] = qnan; of[PC_NEAR] = inf; of[PC_NEAR_T] = qnan; of[PC_LAST_T_A] = qnan;
                of[PC_LAST_T_B] = qnan; of[PC_MAX_STEP] = 0.0;
            }
            continue;
        }
        const long long a0 = sa.off[ia], na = sa.off[ia + 1] - a0;
        const long long b0 = sb.off[ib], nb = sb.off[ib + 1] - b0;
        const double* ta = sa.planes + a0;
        const double* tb = sb.planes + b0;
        PcAcc acc = {inf, inf, inf, 0.0, PC_NONE, PC_NONE, 0};
        for (long long e = threadIdx.x; e < na + nb; e += blockDim.x) {
            const int side = e >= na;
            const long long r = side ? e - na : e;
            const PcSide& own = side ? sb : sa;
            const long long k = (side ? b0 : a0) + r;
            const double t = own.planes[k];
            const long long h = side ? a0 + pc_held(ta, na, t) : b0 + pc_held(tb, nb, t);
            const PcPose me = pc_pose(own.planes, own.R, k, own.hl, own.hw);
            const PcPose other = side ? pc_pose(sa.planes, sa.R, h, sa.hl, sa.hw) : pc_pose(sb.planes, sb.R, h, sb.hl, sb.hw);
            const double d = side ? pc_signed_distance(other, me) : pc_signed_distance(me, other);
            const long long key = ((long long)side << 62) | r;
            if (d < min_gap) {
                acc.count++;
                if (pc_key_less(t, key, acc.first_t, acc.first_k)) { acc.first_t = t; acc.first_k = key; }
            }
            if (d < acc.near || (d == acc.near && pc_key_less(t, key, acc.near_t, acc.near_k))) {
                acc.near = d; acc.near_t = t; acc.near_k = key;
            }
            if (r > 0) acc.step = fmax(acc.step, pc_corner_step(me, pc_pose(own.planes, own.R, k - 1, own.hl, own.hw)));
        }
        for (int o = 16; o > 0; o >>= 1) pc_merge(acc, pc_shfl(acc, o));
        const int warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
        if ((threadIdx.x & 31) == 0) part[warp] = acc;
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < nw; w++) pc_merge(acc, part[w]);
            const bool hit = acc.first_k != PC_NONE;
            oi[PC_STATUS] = PC_OK;
            oi[PC_EVENTS] = na + nb;
            oi[PC_FIRST_SIDE] = hit ? (acc.first_k >> 62) : -1;
            oi[PC_FIRST_ROW] = hit ? (acc.first_k & ((1LL << 62) - 1)) : -1;
            oi[PC_CONTACTS] = acc.count;
            oi[PC_NEAR_SIDE] = acc.near_k >> 62;
            oi[PC_NEAR_ROW] = acc.near_k & ((1LL << 62) - 1);
            of[PC_FIRST_T] = hit ? acc.first_t : qnan;
            of[PC_NEAR] = acc.near;
            of[PC_NEAR_T] = acc.near_t;
            of[PC_LAST_T_A] = ta[na - 1];
            of[PC_LAST_T_B] = tb[nb - 1];
            of[PC_MAX_STEP] = acc.step;
        }
        __syncthreads();                                               // part[] is reused by the next pair
    }
}
