// vap_kernels.cu -- sm_100a kernels + C ABI (include/vap.h) of the batched spline -> motion-profile engine.
//
// Compile: nvcc -O3 -gencode arch=compute_100a,code=sm_100a -lineinfo -fmad=false -shared -Xcompiler -fPIC
// (-fmad=false is load-bearing: the reference never fuses multiply-add, see vap_device.cuh).
//
// Layout: everything is path-major ([B][cap] rows).  Sample-parallel kernels (tables, distance sampling)
// index the fastest dimension with threadIdx.x, so global accesses coalesce; the serial per-path chains
// (velocity passes, time loop) stream along their own row and rely on L1 sector reuse.
#include <cuda_runtime.h>
#include <cstdio>
#include <cstring>
#include <cstdlib>

#include "../../include/vap.h"
#include "vap_device.cuh"
#include "vap_velocity.cuh"
#include "vap_timeloop.cuh"
#include "vap_format.cuh"
#include "vap_parse.cuh"
#include "vap_footprint.cuh"

static thread_local char g_err[512] = "";
static int set_err(const char* where, cudaError_t e)
{
    snprintf(g_err, sizeof(g_err), "%s: %s", where, cudaGetErrorString(e));
    return -100;
}
static int arg_err(const char* msg)
{
    snprintf(g_err, sizeof(g_err), "%s", msg);
    return -101;
}
#define CHECK_LAUNCH(name)                                   \
    do {                                                     \
        cudaError_t e__ = cudaGetLastError();                \
        if (e__ != cudaSuccess) return set_err(name, e__);   \
    } while (0)

extern "C" int vap_version(void) { return 100; }
extern "C" const char* vap_last_error(void) { return g_err; }

// =====================================================================================================
// S0  fit one run of control points (quintic_hermite_spline.py:30-219, :719-736)
//   control points / tangent flags are read with a stride so that the same code serves node tables
//   (stride 12) and stand-alone splines (stride 2).  scratch: dist[n], fd[n][2], sd[n][2] (5n doubles).
// =====================================================================================================
struct RunView {
    const double* px; const double* py; int stride;       // control points
    const int* has; int has_stride, in_mask, out_mask;    // per-node flag word + which bits mean in / out set
    const double* tin; const double* tout;                // [n][2] user tangents already scaled by magnitudes
};

__device__ void fit_run(int n, const RunView& R, bool have_start, double stx, double sty, bool have_end,
                        double etx, double ety, double* __restrict__ seg, double* __restrict__ seglen,
                        double* __restrict__ params_out, double* __restrict__ param_end,
                        double* __restrict__ scratch, bool start_attr, bool end_attr,
                        const double* __restrict__ deriv_in = nullptr, double* __restrict__ deriv_out = nullptr)
{
    // have_start / have_end: a valid boundary tangent is applied to the segment table (:129-132, :543-590);
    // start_attr / end_attr: the attribute "is not None", which is what _compute_derivatives tests (:170,:181);
    // deriv_in: caller-provided first/second derivatives [n][4] (fit(..., first_derivatives, second_derivatives)).
    double* dist = scratch;
    double* fd = scratch + n;
    double* sd = scratch + 3 * n;
#define PX(i) R.px[(size_t)(i) * R.stride]
#define PY(i) R.py[(size_t)(i) * R.stride]
    // _compute_parameters: cumulative chord length (sequential np.cumsum), normalised to [0, n-1]
    double c = 0.0;
    if (params_out) params_out[0] = 0.0;
    for (int i = 0; i < n - 1; i++) {
        double d = norm_ax1(PX(i + 1) - PX(i), PY(i + 1) - PY(i));
        dist[i] = d;
        c = c + d;
        if (params_out) params_out[i + 1] = c;
    }
    double clast = c;
    if (params_out) {
        if (clast == 0.0) {
            for (int i = 0; i < n; i++) params_out[i] = (double)i;
        } else {
            for (int i = 0; i < n; i++) params_out[i] = params_out[i] * (double)(n - 1) / clast;
        }
    }
    *param_end = (clast == 0.0) ? (double)(n - 1) : clast * (double)(n - 1) / clast;
    // _compute_derivatives
    for (int i = 0; i < n; i++) {
        double fx, fy;
        if (i == 0) {
            double cx = PX(1) - PX(0), cy = PY(1) - PY(0);
            if (n == 2 && end_attr) { fx = cx; fy = cy; }
            else { fx = cx / dist[0]; fy = cy / dist[0]; }
        } else if (i == n - 1) {
            double cx = PX(n - 1) - PX(n - 2), cy = PY(n - 1) - PY(n - 2);
            if (n == 2 && start_attr) { fx = cx; fy = cy; }
            else { fx = cx / dist[n - 2]; fy = cy / dist[n - 2]; }
        } else {
            double ax = (PX(i) - PX(i - 1)) / dist[i - 1], ay = (PY(i) - PY(i - 1)) / dist[i - 1];
            double bx = (PX(i + 1) - PX(i)) / dist[i], by = (PY(i + 1) - PY(i)) / dist[i];
            fx = (ax + bx) / 2; fy = (ay + by) / 2;
        }
        fd[2 * i] = fx; fd[2 * i + 1] = fy;
    }
    for (int i = 0; i < n; i++) {
        double sx = 0.0, sy = 0.0;
        if (i > 0 && i < n - 1) {
            double avg = (dist[i - 1] + dist[i]) / 2;
            double den = avg * 0.5;
            sx = (fd[2 * (i + 1)] - fd[2 * (i - 1)]) / den;
            sy = (fd[2 * (i + 1) + 1] - fd[2 * (i - 1) + 1]) / den;
        }
        sd[2 * i] = sx; sd[2 * i + 1] = sy;
    }
    if (deriv_in) {
        for (int i = 0; i < n; i++) {
            fd[2 * i] = deriv_in[4 * i]; fd[2 * i + 1] = deriv_in[4 * i + 1];
            sd[2 * i] = deriv_in[4 * i + 2]; sd[2 * i + 1] = deriv_in[4 * i + 3];
        }
    }
    // segment tables
    for (int i = 0; i < n - 1; i++) {
        double* s = seg + (size_t)i * 12;
        double x0 = PX(i), y0 = PY(i), x1 = PX(i + 1), y1 = PY(i + 1);
        double L = norm1d(x1 - x0, y1 - y0);
        if (seglen) seglen[i] = L;
        s[0] = x0; s[1] = y0; s[2] = x1; s[3] = y1;
        if (L > 0) {
            // reference: L**2 through libm pow, which differs from the correctly rounded L*L by 1 ulp for
            // 0.08 % of inputs (DESIGN.md "known last-bit deviations")
            double L2 = L * L;
            s[4] = fd[2 * i] * L; s[5] = fd[2 * i + 1] * L;
            s[6] = fd[2 * (i + 1)] * L; s[7] = fd[2 * (i + 1) + 1] * L;
            s[8] = sd[2 * i] * L2; s[9] = sd[2 * i + 1] * L2;
            s[10] = sd[2 * (i + 1)] * L2; s[11] = sd[2 * (i + 1) + 1] * L2;
            if (R.has[(size_t)i * R.has_stride] & R.out_mask) { s[4] = R.tout[2 * i]; s[5] = R.tout[2 * i + 1]; }
            if (R.has[(size_t)(i + 1) * R.has_stride] & R.in_mask) { s[6] = R.tin[2 * (i + 1)]; s[7] = R.tin[2 * (i + 1) + 1]; }
        } else {
            s[4] = fd[2 * i]; s[5] = fd[2 * i + 1];
            s[6] = fd[2 * (i + 1)]; s[7] = fd[2 * (i + 1) + 1];
            s[8] = sd[2 * i]; s[9] = sd[2 * i + 1];
            s[10] = sd[2 * (i + 1)]; s[11] = sd[2 * (i + 1) + 1];
        }
    }
    // starting tangent lands on the LAST segment's row 2 (quintic_hermite_spline.py:561), ending on row 3
    double* last = seg + (size_t)(n - 2) * 12;
    if (have_start) { last[4] = stx; last[5] = sty; fd[0] = stx; fd[1] = sty; }
    if (have_end) { last[6] = etx; last[7] = ety; fd[2 * (n - 1)] = etx; fd[2 * (n - 1) + 1] = ety; }
    if (deriv_out) {
        for (int i = 0; i < n; i++) {
            deriv_out[4 * i] = fd[2 * i]; deriv_out[4 * i + 1] = fd[2 * i + 1];
            deriv_out[4 * i + 2] = sd[2 * i]; deriv_out[4 * i + 3] = sd[2 * i + 1];
        }
    }
#undef PX
#undef PY
}

// S0  build_path: one thread per path (spline_manager.py:42-172).  scratch per path: 9*N_max doubles.
__global__ void k_build_path(long long B, int N_max, const double* __restrict__ node_attr,
                             const int* __restrict__ node_flags, const int* __restrict__ n_nodes,
                             double* __restrict__ seg, int* __restrict__ first_node, double* __restrict__ param_end,
                             double* __restrict__ seglen, int* __restrict__ n_splines, int* __restrict__ status,
                             double* __restrict__ scratch, double* __restrict__ params, double* __restrict__ derivs)
{
    long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    int n = n_nodes[b];
    double* pr = params ? params + (size_t)b * 2 * N_max : nullptr;     // concatenated spline.parameters
    double* dv = derivs ? derivs + (size_t)b * 2 * N_max * 4 : nullptr; // concatenated first/second derivatives
    int pc = 0;
    const double* na = node_attr + (size_t)b * N_max * NA;
    const int* nf = node_flags + (size_t)b * N_max;
    double* sg = seg + (size_t)b * (N_max - 1) * 12;
    int* fn = first_node + (size_t)b * (N_max + 1);
    double* pe = param_end + (size_t)b * N_max;
    double* sl = seglen + (size_t)b * N_max;
    double* scr = scratch + (size_t)b * N_max * 9;
    double* tin = scr + 5 * (size_t)N_max;      // node.tangent * magnitude (spline_manager.py:67-73)
    double* tout = tin + 2 * (size_t)N_max;
    n_splines[b] = 0;
    if (n < 2 || n > N_max) { status[b] = ST_FALSE; return; }
    for (int i = 0; i < n; i++) {
        const double* a = na + (size_t)i * NA;
        tin[2 * i] = a[A_TX] * a[A_INMAG]; tin[2 * i + 1] = a[A_TY] * a[A_INMAG];
        tout[2 * i] = a[A_TX] * a[A_OUTMAG]; tout[2 * i + 1] = a[A_TY] * a[A_OUTMAG];
    }
    int S = 0, cur = 0, st = ST_OK;
    bool have_start = false;
    double stx = 0, sty = 0;
    fn[0] = 0;
    for (int i = 1; i < n; i++) {
        const double* a = na + (size_t)i * NA;
        bool rev = (nf[i] & F_REVERSE) != 0;
        bool turn = a[A_TURN] != 0;
        if (!(rev || turn || i == n - 1)) continue;
        bool use_start = have_start;
        double usx = stx, usy = sty;
        have_start = false;
        bool have_end = false;
        double etx = 0, ety = 0;
        if (rev || turn) {
            if (i >= n - 1) { st = ST_INDEX; break; }     // points[i + 1] (spline_manager.py:97)
            double x0 = na[(size_t)(i - 1) * NA + A_X], y0 = na[(size_t)(i - 1) * NA + A_Y];
            double x1 = a[A_X], y1 = a[A_Y];
            double x2 = na[(size_t)(i + 1) * NA + A_X], y2 = na[(size_t)(i + 1) * NA + A_Y];
            double dxp = x1 - x0, dyp = y1 - y0, dxn = x2 - x1, dyn = y2 - y1;
            double prev_len = norm1d(dxp, dyp), next_len = norm1d(dxn, dyn);
            double sp = prev_len > 0 ? 1.0 / prev_len : 1.0;
            double sn = next_len > 0 ? 1.0 / next_len : 1.0;
            double pvx = dxp * sp, pvy = dyp * sp, nvx = dxn * sn, nvy = dyn * sn;
            double min_len = pymin(prev_len, next_len);
            bool has_t = (nf[i] & F_TANGENT) != 0;
            if (turn) {
                double cs = a[A_RCOS], sn2 = a[A_RSIN];
                double ntx = fma(cs, pvx, (-sn2) * pvy);        // rotation_matrix @ prev_vector (BLAS fuses)
                double nty = fma(sn2, pvx, cs * pvy);
                ntx = ntx * min_len; nty = nty * min_len;
                pvx = pvx * min_len; pvy = pvy * min_len;
                if (has_t) {
                    pvx = a[A_TX] * a[A_INMAG]; pvy = a[A_TY] * a[A_INMAG];
                    double vx = a[A_TX], vy = a[A_TY];
                    double r0 = fma(vy, sn2, vx * cs);          // tangent @ rotation_matrix
                    double r1 = fma(vy, cs, vx * (-sn2));
                    ntx = (r0 * -1) * a[A_OUTMAG]; nty = (r1 * -1) * a[A_OUTMAG];
                }
                etx = pvx; ety = pvy; have_end = true;
                stx = ntx; sty = nty; have_start = true;
            } else {
                double dx = pvx - nvx, dy = pvy - nvy;
                double dn = norm1d(dx, dy);
                if (dn > 0) { dx = dx / dn; dy = dy / dn; }
                dx = dx * min_len; dy = dy * min_len;
                if (has_t) { dx = a[A_TX] * a[A_INMAG]; dy = a[A_TY] * a[A_INMAG]; }
                etx = dx; ety = dy; have_end = true;
                stx = -1 * dx; sty = -1 * dy; have_start = true;
                if (has_t) { stx = (-1 * a[A_TX]) * a[A_OUTMAG]; sty = (-1 * a[A_TY]) * a[A_OUTMAG]; }
            }
        }
        int m = i - cur + 1;
        RunView R;
        R.px = na + (size_t)cur * NA + A_X; R.py = na + (size_t)cur * NA + A_Y; R.stride = NA;
        R.has = nf + cur; R.has_stride = 1; R.in_mask = F_TANGENT; R.out_mask = F_TANGENT;
        R.tin = tin + 2 * cur; R.tout = tout + 2 * cur;
        fit_run(m, R, use_start, usx, usy, have_end, etx, ety, sg + (size_t)cur * 12, sl + cur, pr ? pr + pc : nullptr,
                pe + S, scr, use_start, have_end, nullptr, dv ? dv + (size_t)pc * 4 : nullptr);
        pc += m;
        S++;
        fn[S] = i;
        if ((rev || turn) && i < n - 1) cur = i;
    }
    n_splines[b] = (st == ST_OK) ? S : 0;
    status[b] = st;
}

// S0' stand-alone spline fits: one thread per run
__global__ void k_fit_splines(long long Rn, int n_max, const int* __restrict__ n_pts, const double* __restrict__ xy,
                              const int* __restrict__ tan_has, const double* __restrict__ tan_in,
                              const double* __restrict__ tan_out, const int* __restrict__ bnd_has,
                              const double* __restrict__ bnd, double* __restrict__ seg, double* __restrict__ seglen,
                              double* __restrict__ params, int* __restrict__ status, double* __restrict__ scratch,
                              const double* __restrict__ deriv_in, double* __restrict__ deriv_out)
{
    long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= Rn) return;
    int n = n_pts[r];
    if (n < 2 || n > n_max) { status[r] = ST_FALSE; return; }
    RunView R;
    R.px = xy + (size_t)r * n_max * 2; R.py = R.px + 1; R.stride = 2;
    R.has = tan_has + (size_t)r * n_max; R.has_stride = 1; R.in_mask = 1; R.out_mask = 2;
    R.tin = tan_in + (size_t)r * n_max * 2; R.tout = tan_out + (size_t)r * n_max * 2;
    int bh = bnd_has[r];
    const double* bd = bnd + (size_t)r * 4;
    double pe;
    fit_run(n, R, (bh & 1) != 0, bd[0], bd[1], (bh & 2) != 0, bd[2], bd[3], seg + (size_t)r * (n_max - 1) * 12,
            seglen + (size_t)r * n_max, params + (size_t)r * n_max, &pe, scratch + (size_t)r * n_max * 5,
            (bh & 4) != 0, (bh & 8) != 0, (bh & 16) ? deriv_in + (size_t)r * n_max * 4 : nullptr,
            deriv_out ? deriv_out + (size_t)r * n_max * 4 : nullptr);
    status[r] = ST_OK;
}

// evaluation queries
__global__ void k_eval(long long n, const int* __restrict__ path, const double* __restrict__ t, int which, int N_max,
                       const double* __restrict__ seg, const int* __restrict__ first_node,
                       const double* __restrict__ param_end, const int* __restrict__ n_splines,
                       double* __restrict__ out)
{
    long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    PathGeo g = path_geo(path[q], N_max, seg, first_node, param_end, n_splines);
    double ox = 0, oy = 0;
    if (g.S > 0) {
        if (which == 0) eval_path<0>(g, t[q], ox, oy);
        else if (which == 1) eval_path<1>(g, t[q], ox, oy);
        else if (which == 2) eval_path<2>(g, t[q], ox, oy);
        else {
            double dx, dy, ddx, ddy;
            eval_path_d12(g, t[q], dx, dy, ddx, ddy);
            // Spline.get_heading / get_curvature (spline.py:48-80): den = (dx**2 + dy**2) ** 1.5, 0 if |den| < 1e-10
            double s2 = dx * dx + dy * dy;
            double den = s2 * sqrt(s2);
            ox = atan2(dy, dx);
            oy = (fabs(den) < 1e-10) ? 0.0 : (dx * ddy - dy * ddx) / den;
        }
    }
    out[2 * q] = ox; out[2 * q + 1] = oy;
}

// =====================================================================================================
// S1  build_lookup_table: one CTA per path, splines in sequence (the distance offset chains through them);
//     derivative magnitudes in parallel into shared memory, then ONE thread runs the sequential np.cumsum
//     (floating-point addition order is part of the result).
// =====================================================================================================
__global__ void __launch_bounds__(256) k_build_lut(int N_max, const double* __restrict__ seg,
                                                   const int* __restrict__ first_node,
                                                   const double* __restrict__ param_end,
                                                   const int* __restrict__ n_splines, int* __restrict__ status,
                                                   int samples, long long Q_cap, double* __restrict__ lut_d,
                                                   double* __restrict__ lut_t, double* __restrict__ total_len)
{
    extern __shared__ double sm[];   // [2 * samples]: magnitudes / cumulative sums, trapezoid increments
    long long b = blockIdx.x;
    PathGeo g = path_geo(b, N_max, seg, first_node, param_end, n_splines);
    double* od = lut_d + (size_t)b * Q_cap;
    double* ot = lut_t + (size_t)b * Q_cap;
    const int st = status[b];
    const bool too_many = (long long)g.S * samples > Q_cap;     // more splines than the caller's max_splines
    if (st != ST_OK || g.S <= 0 || too_many) {
        __syncthreads();                                         // every thread has read status[b] before it changes
        if (threadIdx.x == 0) {
            total_len[b] = 0.0;
            // the row cannot hold this path's table: a capacity failure the caller retries, never a silent empty path
            if (st == ST_OK && too_many) status[b] = ST_CAPACITY;
        }
        return;
    }
    double current = 0.0, prev_param = 0.0;
    for (int k = 0; k < g.S; k++) {
        int f0 = g.first[k], nseg = g.first[k + 1] - f0;
        double p1 = g.pend[k];
        const double* sg = g.seg + (size_t)f0 * 12;
        double step = (p1 - 0.0) / (double)(samples - 1);      // np.linspace
        double lp1 = (samples > 2) ? 1.0 * step : p1;
        double dtp = lp1 - 0.0;                                 // local_params[1] - local_params[0]
        for (int j = threadIdx.x; j < samples; j += blockDim.x) {
            double lp = (j == samples - 1) ? p1 : (double)j * step;
            double dx, dy;
            eval_spline<1>(sg, nseg, p1, lp, dx, dy);
            sm[j] = norm_ax1(dx, dy);
        }
        __syncthreads();
        // trapezoid increments in parallel (same operations as the reference's vector expression), so that the serial
        // np.cumsum chain below is one dependent addition per entry
        double* inc = sm + samples;
        for (int j = threadIdx.x + 1; j < samples; j += blockDim.x) inc[j] = (sm[j - 1] + sm[j]) * 0.5 * dtp;
        __syncthreads();
        if (threadIdx.x == 0) {
            double c = 0.0;
            sm[0] = 0.0;
            int j = 1;
            for (; j + 8 <= samples; j += 8) {           // eight increments in registers ahead of the dependent additions
                double a[8];
#pragma unroll
                for (int q = 0; q < 8; q++) a[q] = inc[j + q];
#pragma unroll
                for (int q = 0; q < 8; q++) { c = c + a[q]; sm[j + q] = c; }
            }
            for (; j < samples; j++) { c = c + inc[j]; sm[j] = c; }
        }
        __syncthreads();
        for (int j = threadIdx.x; j < samples; j += blockDim.x) {
            double lp = (j == samples - 1) ? p1 : (double)j * step;
            od[(size_t)k * samples + j] = sm[j] + current;
            ot[(size_t)k * samples + j] = lp + prev_param;
        }
        current = sm[samples - 1] + current;
        prev_param += p1 - 0.0;
        __syncthreads();
    }
    if (threadIdx.x == 0) total_len[b] = current;
}

// inverse index of the distance table (see distance_to_time_inv): one CTA per path, one binary search per bucket
__global__ void __launch_bounds__(256) k_build_lut_index(const int* __restrict__ n_splines, const int* __restrict__ status,
                                                         int samples, long long Q_cap, const double* __restrict__ lut_d,
                                                         const double* __restrict__ total_len, int* __restrict__ lut_inv)
{
    const long long b = blockIdx.x;
    int* row = lut_inv + (size_t)b * (Q_cap + LUT_INV_HDR + 2);
    const int S = n_splines[b];
    if (status[b] != ST_OK || S <= 0 || (long long)S * samples > Q_cap) return;
    const int Q = S * samples;
    const double* ld = lut_d + (size_t)b * Q_cap;
    const double L = total_len[b];
    const double scale = (L > 0.0) ? (double)Q / L : 0.0;
    if (threadIdx.x == 0) { row[0] = __double2loint(scale); row[1] = __double2hiint(scale); }
    for (int m = threadIdx.x; m <= Q; m += blockDim.x) {
        const double x = (scale > 0.0) ? (double)m / scale : 0.0;
        int lo = 0, hi = Q;
        while (lo < hi) { int mid = (lo + hi) >> 1; if (ld[mid] < x) lo = mid + 1; else hi = mid; }
        row[LUT_INV_HDR + m] = lo > Q - 1 ? Q - 1 : lo;       // exact for the bucket's lower edge; the lookup verifies both ways
    }
}

// =====================================================================================================
// S2  precompute_path_properties: one thread per (path, table entry)
// =====================================================================================================
#ifndef PROPS_PER_THREAD
#define PROPS_PER_THREAD 8     // table entries per thread: the per-path preamble (geometry pointers, the grid step's division) is paid once
#endif
__global__ void __launch_bounds__(256) k_build_props(int N_max, const int* __restrict__ n_nodes,
                                                     const double* __restrict__ seg,
                                                     const int* __restrict__ first_node,
                                                     const double* __restrict__ param_end,
                                                     const int* __restrict__ n_splines,
                                                     const int* __restrict__ status, int spn, long long P_cap,
                                                     double* __restrict__ prop_k, double* __restrict__ prop_h,
                                                     unsigned tiles_x)
{
    const PathTile pt = path_tile(tiles_x);
    const long long b = pt.b;
    const int n = n_nodes[b];
    const int P = spn * n;
    int j = (int)pt.x * (blockDim.x * PROPS_PER_THREAD) + threadIdx.x;
    if (status[b] != ST_OK || j >= P || (long long)P > P_cap) return;
    const PathGeo g = path_geo(b, N_max, seg, first_node, param_end, n_splines);
    const double step = (double)(n - 1) / (double)(P - 1);
    double* pk = prop_k + (size_t)b * P_cap;
    double* ph = prop_h + (size_t)b * P_cap;
#pragma unroll 1
    for (int it = 0; it < PROPS_PER_THREAD && j < P; ++it, j += blockDim.x) {
        const double t = prop_param(j, P, n, step);
        double dx, dy, ddx, ddy, k, h;
        eval_path_d12(g, t, dx, dy, ddx, ddy);
        curv_heading(dx, dy, ddx, ddy, k, h);
        pk[j] = k;
        ph[j] = h;
    }
}

// table queries for the scalar API
__global__ void k_query_tables(long long n, const int* __restrict__ path, const double* __restrict__ x, int what,
                               const int* __restrict__ n_nodes, const int* __restrict__ n_splines, int samples,
                               long long Q_cap, const double* __restrict__ lut_d, const double* __restrict__ lut_t,
                               const double* __restrict__ total_len, int spn, long long P_cap,
                               const double* __restrict__ prop_k, const double* __restrict__ prop_h,
                               double* __restrict__ out)
{
    long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    long long b = path[q];
    int nn = n_nodes[b];
    if (what == 0) {
        long long hint = -1;
        out[q] = distance_to_time(lut_d + (size_t)b * Q_cap, lut_t + (size_t)b * Q_cap, (long long)samples * n_splines[b],
                                  total_len[b], nn, x[q], hint);
    } else {
        long long P = (long long)spn * nn;
        double step = (double)(nn - 1) / (double)(P - 1);
        const double* v = (what == 1 ? prop_h : prop_k) + (size_t)b * P_cap;
        out[q] = snap_gather(v, x[q], P, nn, step, 1.0 / step);
    }
}

// accumulated distance grid: d_0 = 0, d_{i+1} = fl(d_i + dd)  (single serial chain; built once per dd)
__global__ void k_build_dgrid(long long n, double dd, double* __restrict__ dgrid)
{
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    double d = 0.0;
    for (long long i = 0; i < n; i++) { dgrid[i] = d; d += dd; }
}

// number of distance samples: D = #{i : d_i < L} + 1
__global__ void k_count_samples(long long B, const int* __restrict__ status_in, int* __restrict__ status,
                                long long n_grid, const double* __restrict__ dgrid,
                                const double* __restrict__ total_len, long long D_cap, int* __restrict__ n_samples)
{
    long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    if (status_in[b] != ST_OK) { n_samples[b] = 0; return; }
    double L = total_len[b];
    long long lo = 0, hi = n_grid;      // first i with d_i >= L
    while (lo < hi) {
        long long mid = lo + ((hi - lo) >> 1);
        if (dgrid[mid] < L) lo = mid + 1; else hi = mid;
    }
    long long D = lo + 1;
    if (lo >= n_grid) {               // the grid itself is too short to count on: an upper estimate from the length (sizing only)
        const double est = ceil(L / (dgrid[1] - dgrid[0])) + 2.0;
        D = est < 2147483647.0 ? (long long)est : 2147483647LL;
        if (D <= D_cap) D = D_cap + 1;
    }
    if (lo >= n_grid || D > D_cap) { status[b] = ST_CAPACITY; n_samples[b] = (int)(D > 2147483647LL ? 2147483647LL : D); return; }
    n_samples[b] = (int)D;
}

// =====================================================================================================
// S3  distance sampling: one thread per (path, sample)
// =====================================================================================================
__global__ void __launch_bounds__(256) k_dist_sample(const int* __restrict__ n_nodes,
                                                     const int* __restrict__ n_splines,
                                                     const int* __restrict__ status, const double* __restrict__ dgrid,
                                                     int samples, long long Q_cap, const double* __restrict__ lut_d,
                                                     const double* __restrict__ lut_t,
                                                     const double* __restrict__ total_len, int spn, long long P_cap,
                                                     const double* __restrict__ prop_k,
                                                     const double* __restrict__ prop_h, long long D_cap,
                                                     const int* __restrict__ n_samples, double* __restrict__ t_out,
                                                     double* __restrict__ kap, double* __restrict__ th, unsigned tiles_x)
{
    const PathTile pt = path_tile(tiles_x);
    long long b = pt.b;
    long long i = (long long)pt.x * blockDim.x + threadIdx.x;
    if (status[b] != ST_OK) return;
    long long D = n_samples[b];
    if (i >= D) return;
    int n = n_nodes[b];
    double t;
    if (i == D - 1) t = (double)(n - 1);      // distance_to_time(total_dist)
    else {
        long long hint = -1;
        t = distance_to_time(lut_d + (size_t)b * Q_cap, lut_t + (size_t)b * Q_cap, (long long)samples * n_splines[b],
                             total_len[b], n, dgrid[i], hint);
    }
    long long P = (long long)spn * n;
    double step = (double)(n - 1) / (double)(P - 1);
    double k, h;
    snap_gather2(prop_k + (size_t)b * P_cap, prop_h + (size_t)b * P_cap, t, P, n, step, 1.0 / step, k, h);
    size_t o = (size_t)b * D_cap + i;
    t_out[o] = t; kap[o] = k; th[o] = h;
}

// =====================================================================================================
// S3 events + S4 forward + S5 backward: one thread per path, exact serial recurrences
// (motion_profile_generator.py:93-176, 188-314).
// =====================================================================================================
__global__ void __launch_bounds__(64) k_fwd_bwd(long long B, int N_max, int A_max, const double* __restrict__ node_attr,
                                                const int* __restrict__ node_flags, const int* __restrict__ n_nodes,
                                                const double* __restrict__ ap_attr, const int* __restrict__ ap_flags,
                                                const int* __restrict__ n_ap, const double* __restrict__ cons,
                                                const int* __restrict__ status, double dd, double dt, double start_vel,
                                                double end_vel, long long D_cap, const int* __restrict__ n_samples,
                                                const double* __restrict__ tq, const double* __restrict__ kap,
                                                const double* __restrict__ th, double* __restrict__ vel, int E_cap,
                                                double* __restrict__ max_accels, int* __restrict__ bidx,
                                                int* __restrict__ bval, int* __restrict__ n_ev,
                                                double* __restrict__ t_est, int mode)
{
    long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    if (status[b] != ST_OK) { n_ev[2 * b] = 0; n_ev[2 * b + 1] = 0; if (t_est) t_est[b] = 0.0; return; }
    const int n = n_nodes[b];
    const int A = n_ap ? n_ap[b] : 0;
    const double* na = node_attr + (size_t)b * N_max * NA;
    const int* nf = node_flags + (size_t)b * N_max;
    const double* apa = ap_attr + (size_t)b * A_max * APA;
    const int* apf = ap_flags + (size_t)b * A_max;
    const double V = cons[b * 6 + 0], A0 = cons[b * 6 + 1], w = cons[b * 6 + 5];
    const long long D = n_samples[b];
    const double* T = tq + (size_t)b * D_cap;
    const double* K = kap + (size_t)b * D_cap;
    const double* H = th + (size_t)b * D_cap;
    double* vv = vel + (size_t)b * D_cap;
    double* ma = max_accels + (size_t)b * E_cap;
    int* bi = bidx + (size_t)b * E_cap;
    int* bv = bval + (size_t)b * E_cap;

    const double max_angular_vel = 2 * V / w;
    const double max_angular_accel = 2 * A0 / w;
    const double t_end = (double)(n - 1);

    // ---- event machine state (sampling loop :93-167), run one sample ahead of the forward pass
    int node_num = 0, action_idx = 0, n_acc = 0, n_b = 0;
    double max_velocity = (na[A_MAXVEL] > 0) ? na[A_MAXVEL] : V;
    ma[n_acc++] = (na[A_MAXACC] > 0) ? na[A_MAXACC] : A0;
    bi[0] = 0; bv[0] = 0; n_b = 1;

    double acc = A0, dec = cons[b * 6 + 2];
    int bptr = 0;                 // next boundary entry the forward pass has not applied yet
    double prev_ang_vel = 0.0;
    double v_i = start_vel;
    vv[0] = start_vel;
    double t_i = T[0], th_i = H[0];
    // sample 0 goes through the event logic too (nothing can fire: prev_t == t == 0)
    for (long long i = 0; i < D - 1; i++) {
        // --- append sample i+1 (its initial velocity and events)
        double v0n, t_n = T[i + 1], th_n = H[i + 1];
        if (i + 1 < D - 1) {
            v0n = max_velocity;
            if (frac1(t_i) > frac1(t_n) && t_n < t_end) {
                node_num += 1;
                const double* a = na + (size_t)node_num * NA;
                if (nf[node_num] & F_STOP) v0n = 0.01;
                max_velocity = (a[A_MAXVEL] > 0) ? a[A_MAXVEL] : V;
                ma[n_acc++] = (a[A_MAXACC] > 0) ? a[A_MAXACC] : A0;
                if (node_num < n - 1) {
                    if (bi[n_b - 1] == (int)(i + 1)) bv[n_b - 1] = n_acc - 1;
                    else { bi[n_b] = (int)(i + 1); bv[n_b] = n_acc - 1; n_b++; }
                }
            }
            if (action_idx < A && t_i < apa[action_idx * APA + P_T] && t_n >= apa[action_idx * APA + P_T]) {
                const double* p = apa + (size_t)action_idx * APA;
                max_velocity = (p[P_MAXVEL] > 0) ? p[P_MAXVEL] : V;
                if (apf[action_idx] & F_STOP) v0n = 0.01;
                ma[n_acc++] = (p[P_MAXACC] > 0) ? p[P_MAXACC] : A0;
                if (bi[n_b - 1] == (int)(i + 1)) bv[n_b - 1] = n_acc - 1;
                else { bi[n_b] = (int)(i + 1); bv[n_b] = n_acc - 1; n_b++; }
                action_idx += 1;
            }
        } else {
            v0n = end_vel;
        }
        // --- forward step i -> i+1 (:193-249)
        if (bptr < n_b && bi[bptr] == (int)i) { acc = ma[bv[bptr]]; dec = acc; bptr++; }
        double k = K[i], ak = fabs(k);
        double ang_vel = v_i * ak;
        double vlim, a;
        if (ak < 1e-6) { vlim = V; a = acc; }
        else {
            double dth = th_n - th_i;
            double accel_ang = (ang_vel * ang_vel - prev_ang_vel * prev_ang_vel) / (2 * fabs(dth));
            double v_ang = max_angular_vel / ak;
            double v_kin = 2 * V / (w * ak + 2);
            double v_curve = max_speed_at_curvature(V, w, ak);
            vlim = pymin(pymin(v_ang, v_kin), v_curve);
            double a_ang = max_angular_accel / ak;
            double a_kin = 2 * acc / (w * ak + 2);
            double a_wheel = wheel_accel(acc, fabs(accel_ang), w);
            if (a_wheel < 0) a_wheel = 0;
            a = pymin(pymin(pymin(a_ang, a_kin), a_wheel), acc);
        }
        double next_vel = pymin(vlim, sqrt(v_i * v_i + 2 * a * dd));
        double vn = pymin(v0n, next_vel);
        prev_ang_vel = ang_vel;
        vn = pymin(vn, fabs(V / (1 + (w * ak / 2))));
        vv[i + 1] = vn;
        v_i = vn; t_i = t_n; th_i = th_n;
    }
    ma[n_acc++] = A0;             // :176
    n_ev[2 * b] = n_acc; n_ev[2 * b + 1] = n_b;
    if (mode == 1) { if (t_est) t_est[b] = 0.0; return; }

    // ---- backward pass (:251-311)
    vv[D - 1] = end_vel;
    prev_ang_vel = 0.0;
    v_i = end_vel;
    int bp = n_b - 1;
    double est = 0.0;
    for (long long i = D - 1; i > 0; i--) {
        while (bp >= 0 && bi[bp] > (int)i) bp--;
        if (bp >= 0 && bi[bp] == (int)i) { acc = ma[bv[bp] + 1]; bp--; }
        double k = K[i], ak = fabs(k);
        double ang_vel = v_i * ak;
        double vlim, dcl;
        if (ak < 1e-6) { vlim = V; dcl = dec; }
        else {
            double dth = H[i - 1] - H[i];
            double accel_ang = (ang_vel * ang_vel - prev_ang_vel * prev_ang_vel) / (2 * fabs(dth));
            double v_ang = max_angular_vel / ak;
            double v_kin = 2 * V / (w * ak + 2);
            double v_curve = max_speed_at_curvature(V, w, ak);
            vlim = pymin(pymin(v_ang, v_kin), v_curve);
            double d_ang = max_angular_accel / ak;
            double d_kin = 2 * dec / (w * ak + 2);
            double a_wheel = wheel_accel(acc, accel_ang, w);
            if (a_wheel < 0) a_wheel = 0;
            dcl = pymin(pymin(pymin(d_ang, d_kin), a_wheel), dec);
        }
        double pv = sqrt(v_i * v_i + 2 * dcl * dd);
        pv = pymin(pymin(pv, vv[i - 1]), vlim);
        prev_ang_vel = ang_vel;
        pv = pymin(pv, fabs(V / (1 + (w * ak / 2))));
        vv[i - 1] = pv;
        // travel-time estimate for sizing the time-domain outputs (not part of the reference)
        double vm = 0.5 * (pv + v_i);
        est += dd / ((vm > 0.05 ? vm : 0.05) * dt);
        v_i = pv;
    }
    if (t_est) {
        // inserts: waits and turn profiles of every node / action point (upper bound: assume all fire)
        double extra = 0.0;
        for (int i = 0; i < n; i++) {
            const double* a = na + (size_t)i * NA;
            if (a[A_WAIT] > 0) extra += floor(a[A_WAIT] / dt);
            if (a[A_TURN] != 0) {
                double angle = a[A_TURN] * (VAP_PI / 180.0);
                Trapezoid tz = trapezoid_setup(V, A0, fabs(angle) * w / 2, dt);
                extra += (double)tz.K;
            }
        }
        for (int i = 0; i < A; i++) if (apa[i * APA + P_WAIT] > 0) extra += floor(apa[i * APA + P_WAIT] / dt);
        t_est[b] = est + extra;
    }
}

// =====================================================================================================
// S6  time-domain stage + S7 summary: one thread per path (motion_profile_generator.py:414-628)
// =====================================================================================================
struct OutRows {
    double *tm, *pos, *lin, *acc, *head, *ang, *x, *y;
    long long cap, T;
    __device__ __forceinline__ void push(double t, double p, double l, double a, double h, double w, double xx, double yy)
    {
        if (T < cap) { tm[T] = t; pos[T] = p; lin[T] = l; acc[T] = a; head[T] = h; ang[T] = w; x[T] = xx; y[T] = yy; }
        T++;
    }
};

__global__ void __launch_bounds__(64) k_resample(long long B, int N_max, int A_max, const double* __restrict__ node_attr,
                                                 const int* __restrict__ node_flags, const int* __restrict__ n_nodes,
                                                 const double* __restrict__ ap_attr, const int* __restrict__ ap_flags,
                                                 const int* __restrict__ n_ap, const double* __restrict__ cons,
                                                 int* __restrict__ status, double dt, double dd,
                                                 const double* __restrict__ seg, const int* __restrict__ first_node,
                                                 const double* __restrict__ param_end,
                                                 const int* __restrict__ n_splines, int samples, long long Q_cap,
                                                 const double* __restrict__ lut_d, const double* __restrict__ lut_t,
                                                 const double* __restrict__ total_len, int spn, long long P_cap,
                                                 const double* __restrict__ prop_k, const double* __restrict__ prop_h,
                                                 long long D_cap, const int* __restrict__ n_samples,
                                                 const double* __restrict__ vel, long long T_cap,
                                                 double* __restrict__ out, int* __restrict__ nodes_map,
                                                 int* __restrict__ actions_map, int* __restrict__ n_maps,
                                                 int* __restrict__ n_out, double* __restrict__ summary,
                                                 long long oplane, int only_status)
{
    long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    int st = status[b];
    // only_status != 0: the pass that redoes, reference-shaped, the paths the split time stage gave up on (status ==
    // only_status, i.e. ST_EVENTS: a position that oscillates across an action point or a node more often than the
    // candidate tables hold); every other path leaves untouched
    if (only_status != 0) { if (st != only_status) return; st = ST_OK; }
    const double L = total_len[b];
    int* nmap = nodes_map + (size_t)b * (N_max + 1);
    int* amap = actions_map + (size_t)b * (A_max > 0 ? A_max : 1);
    int nm = 0, am = 0;
    OutRows o;
    size_t plane = oplane > 0 ? (size_t)oplane : (size_t)B * T_cap;
    o.tm = out + (size_t)b * T_cap; o.pos = o.tm + plane; o.lin = o.pos + plane; o.acc = o.lin + plane;
    o.head = o.acc + plane; o.ang = o.head + plane; o.x = o.ang + plane; o.y = o.x + plane;
    o.cap = T_cap; o.T = 0;
    double last_time = 0.0, max_abs_v = 0.0;
    if (st == ST_OK) {
        const int n = n_nodes[b];
        const int A = n_ap ? n_ap[b] : 0;
        const double* na = node_attr + (size_t)b * N_max * NA;
        const int* nf = node_flags + (size_t)b * N_max;
        const double* apa = ap_attr + (size_t)b * A_max * APA;
        const double V = cons[b * 6 + 0], max_acc = cons[b * 6 + 1], max_dec = cons[b * 6 + 2], w = cons[b * 6 + 5];
        PathGeo g = path_geo(b, N_max, seg, first_node, param_end, n_splines);
        const double* ld = lut_d + (size_t)b * Q_cap;
        const double* lt = lut_t + (size_t)b * Q_cap;
        const long long Q = (long long)samples * g.S;
        const long long P = (long long)spn * n;
        const double pstep = (double)(n - 1) / (double)(P - 1), inv_pstep = 1.0 / pstep;
        const double* pk = prop_k + (size_t)b * P_cap;
        const double* ph = prop_h + (size_t)b * P_cap;
        const long long D = n_samples[b];
        const double* vv = vel + (size_t)b * D_cap;
        const double inv_dd = 1.0 / dd;

        double current_time = 0.0, current_pos = 0.0, current_vel = vv[0];
        bool is_reversed = (nf[0] & F_REVERSE) != 0;
        nmap[nm++] = 0;
        double last_pos = 0.0, last_head = 0.0, last_x = 0.0, last_y = 0.0;   // [-1] entries of the result lists
        bool have_rows = false;
        if (na[A_TURN] != 0) st = ST_INDEX;          // headings[-1] on an empty list (:440)
        if (st == ST_OK && na[A_WAIT] > 0) {          // :459-476
            long long steps = (long long)(na[A_WAIT] / dt);
            if (!(na[A_WAIT] / dt < (double)VAP_ROW_LIMIT)) { st = ST_DIVERGED; steps = 0; }
            double h = -1 * snap_gather(ph, 0.0, P, n, pstep, inv_pstep);
            if (is_reversed) h -= VAP_PI;
            if (h > VAP_PI) h -= 2 * VAP_PI;
            if (h < -VAP_PI) h += 2 * VAP_PI;
            double px, py;
            eval_path<0>(g, 0.0, px, py);
            for (long long i = 0; i < steps; i++) o.push(current_time + (double)i * dt, 0.0, 0.0, 0.0, h, 0.0, px, py);
            current_time += (double)steps * dt;
            if (steps > 0) { last_head = h; last_x = px; last_y = py; have_rows = true; }
        }
        double prev_t = 0.0;
        int action_idx = 0, node_idx = 0;
        const double end_param = (double)(n - 1);
        long long hint = -1;
        while (st == ST_OK && current_pos < L) {
            if (o.T >= 16 * T_cap + 1000000 || o.T >= VAP_ROW_LIMIT) { st = ST_DIVERGED; break; }   // diverging loop
            double t = distance_to_time(ld, lt, Q, L, n, current_pos, hint);
            if (frac1(t) < frac1(prev_t) && t < end_param) {
                nmap[nm++] = (int)o.T;
                node_idx += 1;
                // spline_manager.nodes[node_idx] (:530) raises IndexError once a position that oscillates across node
                // boundaries (steps that move backwards) has produced more crossings than there are nodes
                if (node_idx >= n) { st = ST_INDEX; break; }
                const double* a = na + (size_t)node_idx * NA;
                if (a[A_TURN] != 0) {                 // handle_turn (:487-507)
                    if (!have_rows) { st = ST_INDEX; break; }
                    double angle = a[A_TURN] * (VAP_PI / 180.0);        // np.radians
                    Trapezoid tz = trapezoid_setup(V, max_acc, fabs(angle) * w / 2, dt);
                    if (!(tz.K < VAP_ROW_LIMIT)) { st = ST_DIVERGED; break; }
                    double sgn = angle > 0 ? -1.0 : 1.0;
                    double accum = 0.0, hprev = 0.0;
                    double start_heading = last_head;
                    for (long long i = 0; i < tz.K; i++) {
                        double v = trapezoid_vel(tz, i, dt);
                        double hraw = (accum / (w / 2)) * sgn;       // motion_profile_angle (:334-339)
                        accum += v * dt;
                        double om = (i == 0) ? 0.0 : (hraw - hprev) / dt;
                        hprev = hraw;
                        double hh = hraw;
                        while (hh + start_heading > VAP_PI) hh -= 2 * VAP_PI;
                        while (hh + start_heading < -VAP_PI) hh += 2 * VAP_PI;
                        last_head = start_heading + hh;
                        o.push(current_time + (double)i * dt, last_pos, 0.0, 0.0, last_head, om, last_x, last_y);
                    }
                    current_time = current_time + (double)tz.K * dt;
                }
                if (nf[node_idx] & F_REVERSE) is_reversed = !is_reversed;
                if (a[A_WAIT] > 0) {                  // handle_wait (:509-518)
                    if (!have_rows) { st = ST_INDEX; break; }
                    if (!(a[A_WAIT] / dt < (double)VAP_ROW_LIMIT)) { st = ST_DIVERGED; break; }
                    long long steps = (long long)(a[A_WAIT] / dt);
                    for (long long i = 0; i < steps; i++)
                        o.push(current_time + (double)i * dt, 0.0, 0.0, 0.0, last_head, 0.0, last_x, last_y);
                    if (steps > 0) last_pos = 0.0;
                    current_time = current_time + (double)steps * dt;
                }
            }
            if (action_idx < A) {
                const double* p = apa + (size_t)action_idx * APA;
                if (prev_t < p[P_T] && p[P_T] < t) {
                    amap[am++] = (int)o.T;
                    if (p[P_WAIT] > 0) {
                        if (!have_rows) { st = ST_INDEX; break; }
                        if (!(p[P_WAIT] / dt < (double)VAP_ROW_LIMIT)) { st = ST_DIVERGED; break; }
                        long long steps = (long long)(p[P_WAIT] / dt);
                        for (long long i = 0; i < steps; i++)
                            o.push(current_time + (double)i * dt, 0.0, 0.0, 0.0, last_head, 0.0, last_x, last_y);
                        if (steps > 0) last_pos = 0.0;
                        current_time = current_time + (double)steps * dt;
                    }
                    action_idx += 1;
                }
            }
            prev_t = t;
            double curvature, heading;
            snap_gather2(pk, ph, t, P, n, pstep, inv_pstep, curvature, heading);
            heading = heading - (is_reversed ? VAP_PI : 0.0);
            heading = pymod_pos(heading + VAP_PI, 2 * VAP_PI) - VAP_PI;
            heading *= -1;
            double cx, cy;
            eval_path<0>(g, t, cx, cy);
            double tv = lerp_uniform(current_pos, dd, inv_dd, D, vv);
            double ntv = lerp_uniform(current_pos + dd, dd, inv_dd, D, vv);
            tv = pymax((tv + ntv) / 2, 0.001);
            double accel = (tv - current_vel) / dt;
            accel = fmin(fmax(accel, -max_dec), max_acc);          // np.clip
            double angular_vel = tv * curvature * -1;
            current_vel = fmin(fmax(current_vel + accel * dt, 0.0), tv);
            double dpos = current_vel * dt + 0.5 * accel * dt * dt;
            if (current_vel <= 0.1) dpos = 0.1 * dt + 0.5 * accel * dt * dt;
            current_pos += dpos;
            double sgn = is_reversed ? -1.0 : 1.0;
            o.push(current_time, current_pos, current_vel * sgn, accel * sgn, heading, angular_vel, cx, cy);
            last_pos = current_pos; last_head = heading; last_x = cx; last_y = cy; have_rows = true;
            last_time = current_time;
            max_abs_v = fmax(max_abs_v, current_vel);
            current_time += dt;
        }
        if (st == ST_OK) nmap[nm++] = (int)o.T;            // gui/path.py:342
        if (st == ST_OK && o.T > T_cap) st = ST_CAPACITY;
    }
    long long T = (st == ST_OK || st == ST_CAPACITY) ? o.T : 0;
    if (T > 0 && T <= T_cap) last_time = o.tm[T - 1];
    if (!(st == ST_OK || st == ST_CAPACITY)) { last_time = 0.0; max_abs_v = 0.0; }     // a failed path has no t_end / max |v|
    n_out[b] = (int)T;
    n_maps[2 * b] = nm; n_maps[2 * b + 1] = am;
    status[b] = st;
    double* sr = summary + (size_t)b * 5;
    sr[0] = (double)T; sr[1] = L; sr[2] = last_time; sr[3] = max_abs_v; sr[4] = (double)st;
}

// =====================================================================================================
// S1' Gauss-Legendre arc length and bisection inverse (quintic_hermite_spline.py:592-717): thread per query
// =====================================================================================================
__device__ __forceinline__ double np_sum(const double* a, int n)
{   // numpy pairwise_sum for n <= 128: 8 accumulators, then the tail
    if (n < 8) { double r = 0.0; for (int i = 0; i < n; i++) r += a[i]; return r; }
    double r[8];
    for (int j = 0; j < 8; j++) r[j] = a[j];
    int i = 8;
    for (; i < n - (n % 8); i += 8) for (int j = 0; j < 8; j++) r[j] += a[i + j];
    double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
    for (; i < n; i++) res += a[i];
    return res;
}
__device__ double gl_arclen(const double* sg, int nseg, double pend, double t0, double t1, int npts,
                            const double* __restrict__ pts, const double* __restrict__ wts)
{
    double half = (t1 - t0) / 2, mid = (t0 + t1) / 2;
    double wm[128];
    for (int j = 0; j < npts; j++) {
        double tau = pts[j] * half + mid;
        double dx, dy;
        eval_spline<1>(sg, nseg, pend, tau, dx, dy);
        wm[j] = wts[j] * norm1d(dx, dy);
    }
    return half * np_sum(wm, npts);
}
__global__ void k_gl(long long n, const int* __restrict__ path, const int* __restrict__ spl, const double* __restrict__ a,
                     const double* __restrict__ bb, int mode, int max_iter, int npts, const double* __restrict__ pts,
                     const double* __restrict__ wts, int N_max, const double* __restrict__ seg,
                     const int* __restrict__ first_node, const double* __restrict__ param_end,
                     double* __restrict__ out, int* __restrict__ qstatus)
{
    long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    long long b = path[q];
    int k = spl[q];
    const int* fn = first_node + (size_t)b * (N_max + 1);
    int f0 = fn[k], nseg = fn[k + 1] - f0;
    double pend = param_end[(size_t)b * N_max + k];
    const double* sg = seg + ((size_t)b * (N_max - 1) + f0) * 12;
    if (mode == 0) {
        double t0 = a[q], t1 = bb[q];
        if (t0 >= t1 || t0 < 0.0 || t1 > pend) { qstatus[q] = ST_VALUE; out[q] = 0.0; return; }
        out[q] = gl_arclen(sg, nseg, pend, t0, t1, npts, pts, wts);
        qstatus[q] = ST_OK;
    } else {
        double s = a[q], tol = bb[q];
        if (s < 0) { qstatus[q] = ST_VALUE; out[q] = 0.0; return; }
        double total = gl_arclen(sg, nseg, pend, 0.0, pend, npts, pts, wts);
        if (s > total) { qstatus[q] = ST_VALUE; out[q] = 0.0; return; }
        qstatus[q] = ST_OK;
        if (s == 0) { out[q] = 0.0; return; }
        if (s == total) { out[q] = pend; return; }
        double lo = 0.0, hi = pend;
        for (int it = 0; it < max_iter; it++) {
            double m = (lo + hi) / 2;
            // get_arc_length(t_start, t_mid) raises if t_mid <= t_start; cannot happen for lo >= 0 < hi
            double len = gl_arclen(sg, nseg, pend, 0.0, m, npts, pts, wts);
            double err = len - s;
            if (fabs(err) < tol) { out[q] = m; return; }
            if (err > 0) hi = m; else lo = m;
        }
        out[q] = (lo + hi) / 2;
    }
}

// motion_profile_angle / generate_trapezoidal_profile: thread per query
__global__ void k_turn_profile(long long n, const double* __restrict__ q, int mode, long long K_cap,
                               double* __restrict__ out_a, double* __restrict__ out_b, int* __restrict__ counts)
{
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double* p = q + (size_t)i * 5;
    double x = p[0], V = p[1], A = p[2], w = p[3], dt = p[4];
    double* oa = out_a + (size_t)i * K_cap;
    if (mode == 1) {
        Trapezoid tz = trapezoid_setup(V, A, x, dt);
        counts[i] = (int)tz.K;
        for (long long j = 0; j < tz.K && j < K_cap; j++) oa[j] = trapezoid_vel(tz, j, dt);
        return;
    }
    double* ob = out_b + (size_t)i * K_cap;
    Trapezoid tz = trapezoid_setup(V, A, fabs(x) * w / 2, dt);
    counts[i] = (int)tz.K;
    double sgn = x > 0 ? -1.0 : 1.0, accum = 0.0, hprev = 0.0;
    for (long long j = 0; j < tz.K && j < K_cap; j++) {
        double v = trapezoid_vel(tz, j, dt);
        double h = (accum / (w / 2)) * sgn;
        accum += v * dt;
        oa[j] = h;
        ob[j] = (j == 0) ? 0.0 : (h - hprev) / dt;
        hprev = h;
    }
}

// lerp (motion_profile_generator.py:349-386), cache=None, general sorted xs
__global__ void k_lerp(long long n, const double* __restrict__ x, long long m, const double* __restrict__ xs,
                       const double* __restrict__ ys, double* __restrict__ out)
{
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double xv = x[i];
    long long lo = 0, hi = m;    // searchsorted side='right'
    while (lo < hi) {
        long long mid = lo + ((hi - lo) >> 1);
        if (xs[mid] <= xv) lo = mid + 1; else hi = mid;
    }
    long long idx = lo - 1;
    if (idx < 0) { out[i] = ys[0]; return; }
    if (idx >= m - 1) { out[i] = ys[m - 1]; return; }
    double x0 = xs[idx], x1 = xs[idx + 1], y0 = ys[idx], y1 = ys[idx + 1];
    out[i] = y0 + (xv - x0) * (y1 - y0) / (x1 - x0);
}

// get_wheel_trajectory (motion_profile_generator.py:631-646)
__global__ void k_wheel(long long n, const double* __restrict__ lin, const double* __restrict__ ang, double tw,
                        double* __restrict__ left, double* __restrict__ right)
{
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double l = lin[i], a = ang[i];
    left[i] = l - (a * tw / 2);
    right[i] = l + (a * tw / 2);
}

// =====================================================================================================
// C ABI
// =====================================================================================================
static inline unsigned blocks_for(long long n, int bs) { return (unsigned)((n + bs - 1) / bs); }
#define STREAM ((cudaStream_t)stream)

extern "C" int vap_build_path(int64_t B, int N_max, const double* node_attr, const int32_t* node_flags,
                              const int32_t* n_nodes, double* seg, int32_t* first_node, double* param_end,
                              double* seglen, int32_t* n_splines, int32_t* status, double* scratch, double* params,
                              double* derivs, void* stream)
{
    if (B <= 0) return 0;
    if (N_max < 2) return arg_err("vap_build_path: N_max < 2");
    k_build_path<<<blocks_for(B, 128), 128, 0, STREAM>>>(B, N_max, node_attr, node_flags, n_nodes, seg, first_node,
                                                        param_end, seglen, n_splines, status, scratch, params, derivs);
    CHECK_LAUNCH("vap_build_path");
    return 0;
}

extern "C" int vap_fit_splines(int64_t R, int n_max, const int32_t* n_pts, const double* xy, const int32_t* tan_has,
                               const double* tan_in, const double* tan_out, const int32_t* bnd_has, const double* bnd,
                               double* seg, double* seglen, double* params, int32_t* status, double* scratch,
                               const double* deriv_in, double* deriv_out, void* stream)
{
    if (R <= 0) return 0;
    if (n_max < 2) return arg_err("vap_fit_splines: n_max < 2");
    k_fit_splines<<<blocks_for(R, 128), 128, 0, STREAM>>>(R, n_max, n_pts, xy, tan_has, tan_in, tan_out, bnd_has, bnd,
                                                         seg, seglen, params, status, scratch, deriv_in, deriv_out);
    CHECK_LAUNCH("vap_fit_splines");
    return 0;
}

extern "C" int vap_eval(int64_t n, const int32_t* path, const double* t, int which, int N_max, const double* seg,
                        const int32_t* first_node, const double* param_end, const int32_t* n_splines, double* out,
                        void* stream)
{
    if (n <= 0) return 0;
    if (which < 0 || which > 3) return arg_err("vap_eval: which must be 0..3");
    k_eval<<<blocks_for(n, 128), 128, 0, STREAM>>>(n, path, t, which, N_max, seg, first_node, param_end, n_splines, out);
    CHECK_LAUNCH("vap_eval");
    return 0;
}

extern "C" int vap_build_lut(int64_t B, int N_max, const double* seg, const int32_t* first_node,
                             const double* param_end, const int32_t* n_splines, int32_t* status, int samples,
                             int64_t Q_cap, double* lut_d, double* lut_t, double* total_len, void* stream)
{
    if (B <= 0) return 0;
    if (samples < 2 || samples > 6000) return arg_err("vap_build_lut: samples must be in [2, 6000]");
    const size_t lut_sm = 2 * (size_t)samples * sizeof(double);
    if (lut_sm > 48 * 1024) cudaFuncSetAttribute(k_build_lut, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lut_sm);
    k_build_lut<<<(unsigned)B, 256, lut_sm, STREAM>>>(N_max, seg, first_node, param_end,
                                                                               n_splines, status, samples, Q_cap,
                                                                               lut_d, lut_t, total_len);
    CHECK_LAUNCH("vap_build_lut");
    return 0;
}

extern "C" int64_t vap_lut_index_row_ints(int64_t Q_cap) { return Q_cap + LUT_INV_HDR + 2; }
extern "C" int vap_build_lut_index(int64_t B, const int32_t* n_splines, const int32_t* status, int samples, int64_t Q_cap,
                                   const double* lut_d, const double* total_len, int32_t* lut_inv, void* stream)
{
    if (B <= 0) return 0;
    k_build_lut_index<<<(unsigned)B, 256, 0, STREAM>>>(n_splines, status, samples, Q_cap, lut_d, total_len, lut_inv);
    CHECK_LAUNCH("vap_build_lut_index");
    return 0;
}

extern "C" int vap_build_props(int64_t B, int N_max, const int32_t* n_nodes, const double* seg,
                               const int32_t* first_node, const double* param_end, const int32_t* n_splines,
                               const int32_t* status, int spn, int64_t P_cap, double* prop_k, double* prop_h,
                               void* stream)
{
    if (B <= 0) return 0;
    const unsigned tx = blocks_for(P_cap, 256 * PROPS_PER_THREAD);
    if ((long long)tx * B > 2147483647LL) return arg_err("vap_build_props: more than 2^31 CTAs (tile the batch)");
    const unsigned grid = tx * (unsigned)B;
    k_build_props<<<grid, 256, 0, STREAM>>>(N_max, n_nodes, seg, first_node, param_end, n_splines, status, spn, P_cap,
                                            prop_k, prop_h, tx);
    CHECK_LAUNCH("vap_build_props");
    return 0;
}

extern "C" int vap_query_tables(int64_t n, const int32_t* path, const double* x, int what, const int32_t* n_nodes,
                                const int32_t* n_splines, int samples, int64_t Q_cap, const double* lut_d,
                                const double* lut_t, const double* total_len, int spn, int64_t P_cap,
                                const double* prop_k, const double* prop_h, double* out, void* stream)
{
    if (n <= 0) return 0;
    k_query_tables<<<blocks_for(n, 128), 128, 0, STREAM>>>(n, path, x, what, n_nodes, n_splines, samples, Q_cap, lut_d,
                                                          lut_t, total_len, spn, P_cap, prop_k, prop_h, out);
    CHECK_LAUNCH("vap_query_tables");
    return 0;
}

extern "C" int vap_build_dgrid(int64_t n, double dd, double* dgrid, void* stream)
{
    if (n <= 0) return 0;
    k_build_dgrid<<<1, 1, 0, STREAM>>>(n, dd, dgrid);
    CHECK_LAUNCH("vap_build_dgrid");
    return 0;
}

extern "C" int vap_build_lerp_recip(int64_t n, double dd, double* rden, void* stream)
{
    if (n <= 0) return 0;
    k_build_lerp_recip<<<blocks_for(n, 256), 256, 0, STREAM>>>(n, dd, rden);
    CHECK_LAUNCH("vap_build_lerp_recip");
    return 0;
}

extern "C" int vap_dist_sample(int64_t B, const int32_t* n_nodes, const int32_t* n_splines, int32_t* status,
                               int64_t n_grid, const double* dgrid, int samples, int64_t Q_cap, const double* lut_d,
                               const double* lut_t, const double* total_len, int spn, int64_t P_cap,
                               const double* prop_k, const double* prop_h, int64_t D_cap, int32_t* n_samples,
                               double* t, double* kap, double* th, void* stream)
{
    if (B <= 0) return 0;
    k_count_samples<<<blocks_for(B, 128), 128, 0, STREAM>>>(B, status, status, n_grid, dgrid, total_len, D_cap, n_samples);
    CHECK_LAUNCH("vap_dist_sample/count");
    const unsigned tx = blocks_for(D_cap, 256);
    if ((long long)tx * B > 2147483647LL) return arg_err("vap_dist_sample: more than 2^31 CTAs (tile the batch)");
    const unsigned grid = tx * (unsigned)B;
    k_dist_sample<<<grid, 256, 0, STREAM>>>(n_nodes, n_splines, status, dgrid, samples, Q_cap, lut_d, lut_t, total_len,
                                            spn, P_cap, prop_k, prop_h, D_cap, n_samples, t, kap, th, tx);
    CHECK_LAUNCH("vap_dist_sample");
    return 0;
}

extern "C" int vap_fwd_bwd(int64_t B, int N_max, int A_max, const double* node_attr, const int32_t* node_flags,
                           const int32_t* n_nodes, const double* ap_attr, const int32_t* ap_flags, const int32_t* n_ap,
                           const double* cons, const int32_t* status, double dd, double dt, double start_vel,
                           double end_vel, int64_t D_cap, const int32_t* n_samples, const double* t, const double* kap,
                           const double* th, double* vel, int E_cap, double* max_accels, int32_t* bidx, int32_t* bval,
                           int32_t* n_ev, double* t_est, int mode, void* stream)
{
    if (B <= 0) return 0;
    if (E_cap < N_max + A_max + 2) return arg_err("vap_fwd_bwd: E_cap < N_max + A_max + 2");
    k_fwd_bwd<<<blocks_for(B, 32), 32, 0, STREAM>>>(B, N_max, A_max, node_attr, node_flags, n_nodes, ap_attr, ap_flags,
                                                   n_ap, cons, status, dd, dt, start_vel, end_vel, D_cap, n_samples, t,
                                                   kap, th, vel, E_cap, max_accels, bidx, bval, n_ev, t_est, mode);
    CHECK_LAUNCH("vap_fwd_bwd");
    return 0;
}

extern "C" int vap_resample(int64_t B, int N_max, int A_max, const double* node_attr, const int32_t* node_flags,
                            const int32_t* n_nodes, const double* ap_attr, const int32_t* ap_flags, const int32_t* n_ap,
                            const double* cons, int32_t* status, double dt, double dd, const double* seg,
                            const int32_t* first_node, const double* param_end, const int32_t* n_splines, int samples,
                            int64_t Q_cap, const double* lut_d, const double* lut_t, const double* total_len, int spn,
                            int64_t P_cap, const double* prop_k, const double* prop_h, int64_t D_cap,
                            const int32_t* n_samples, const double* vel, int64_t T_cap, double* out,
                            int32_t* nodes_map, int32_t* actions_map, int32_t* n_maps, int32_t* n_out, double* summary,
                            void* stream)
{
    if (B <= 0) return 0;
    k_resample<<<blocks_for(B, 32), 32, 0, STREAM>>>(B, N_max, A_max, node_attr, node_flags, n_nodes, ap_attr, ap_flags,
                                                    n_ap, cons, status, dt, dd, seg, first_node, param_end, n_splines,
                                                    samples, Q_cap, lut_d, lut_t, total_len, spn, P_cap, prop_k, prop_h,
                                                    D_cap, n_samples, vel, T_cap, out, nodes_map, actions_map, n_maps,
                                                    n_out, summary, 0, 0);
    CHECK_LAUNCH("vap_resample");
    return 0;
}

extern "C" int vap_gl(int64_t n, const int32_t* path, const int32_t* spl, const double* a, const double* b, int mode,
                      int max_iter, int npts, const double* gl_pts, const double* gl_wts, int N_max, const double* seg,
                      const int32_t* first_node, const double* param_end, double* out, int32_t* qstatus, void* stream)
{
    if (n <= 0) return 0;
    if (npts < 1 || npts > 128) return arg_err("vap_gl: npts must be in [1, 128]");
    k_gl<<<blocks_for(n, 64), 64, 0, STREAM>>>(n, path, spl, a, b, mode, max_iter, npts, gl_pts, gl_wts, N_max, seg,
                                              first_node, param_end, out, qstatus);
    CHECK_LAUNCH("vap_gl");
    return 0;
}

extern "C" int vap_turn_profile(int64_t n, const double* q, int mode, int64_t K_cap, double* out_a, double* out_b,
                                int32_t* counts, void* stream)
{
    if (n <= 0) return 0;
    k_turn_profile<<<blocks_for(n, 64), 64, 0, STREAM>>>(n, q, mode, K_cap, out_a, out_b, counts);
    CHECK_LAUNCH("vap_turn_profile");
    return 0;
}

extern "C" int vap_lerp(int64_t n, const double* x, int64_t m, const double* xs, const double* ys, double* out,
                        void* stream)
{
    if (n <= 0) return 0;
    if (m < 1) return arg_err("vap_lerp: empty table");
    k_lerp<<<blocks_for(n, 128), 128, 0, STREAM>>>(n, x, m, xs, ys, out);
    CHECK_LAUNCH("vap_lerp");
    return 0;
}

extern "C" int vap_wheel_trajectory(int64_t n, const double* lin, const double* ang, double track_width, double* left,
                                    double* right, void* stream)
{
    if (n <= 0) return 0;
    k_wheel<<<blocks_for(n, 256), 256, 0, STREAM>>>(n, lin, ang, track_width, left, right);
    CHECK_LAUNCH("vap_wheel_trajectory");
    return 0;
}

// ---- v2 velocity path ------------------------------------------------------------------------------------------
extern "C" int64_t vap_event_scratch_ints(int64_t B, int N_max, int A_max)
{
    int Am = A_max > 0 ? A_max : 1;
    return B * N_max + B + B * Am * EV_AP_CAND + B * Am;
}

// the event candidates of the sampling kernels in ev_scratch (vap_event_scratch_ints elements, Am = max(A_max, 1)):
// wrap[B][N_max] | nwrap[B] | apc[B][Am][EV_AP_CAND] | napc[B][Am]; the two candidate counters start at zero
struct EventScratch { int32_t *wrap, *nwrap, *apc, *napc; };
static cudaError_t event_scratch(int32_t* ev_scratch, int64_t B, int N_max, int Am, cudaStream_t st, EventScratch& c)
{
    c.wrap = ev_scratch;
    c.nwrap = c.wrap + (size_t)B * N_max;
    c.apc = c.nwrap + B;
    c.napc = c.apc + (size_t)B * Am * EV_AP_CAND;
    cudaError_t e = cudaMemsetAsync(c.nwrap, 0, sizeof(int32_t) * (size_t)B, st);
    if (e != cudaSuccess) return e;
    return cudaMemsetAsync(c.napc, 0, sizeof(int32_t) * (size_t)B * Am, st);
}

// slots per path row of the chunk-interleaved pass arrays (records, override limits, forward velocities): the samples, one
// block of four rows per chunk for rounding the chunk length up, one more for the passes' look-ahead loads, the tail slot
extern "C" int64_t vap_pass_row_slots(int64_t D_cap, int chunks) { return ((D_cap + 8 * (int64_t)chunks + 64 + 1) / 2) * 2; }

template <int NT>
static int launch_passes(int64_t B, size_t ss, cudaStream_t st, const double* cons, const int32_t* status, double dd, double dt,
                         double start_vel, double end_vel, long long RS, long long D_cap, const int32_t* n_samples,
                         const double* rec, int E_cap, const double* max_accels, const int32_t* bidx, const int32_t* bval,
                         const int32_t* n_ev, const int32_t* vr_idx, const double* vr_val, const int32_t* st_idx,
                         const int32_t* n_vr, double* vel_f, double* vel, float* t_est, int32_t* rounds, bool backward,
                         int warm, int max_rounds, const double* statB)
{
    // behind the tables every warp has a two-stage ring of 4 (forward) / 5 (backward) planes of 1 KB + 2 mbarriers
    const int warps = (NT + 31) / 32;
    const int ring_off = (int)((ss + 127) / 128 * 128);
    const int planes = backward ? 5 : 4;
    const size_t smem = (size_t)ring_off + (size_t)warps * (2 * planes * TMA_PLANE_DOUBLES * 8 + 16);
    cudaError_t e = cudaSuccess;
    if (!backward) {
        if (smem > 48 * 1024) e = cudaFuncSetAttribute(k_fwd_chunked<NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return set_err("vap_velocity_profile/attr", e);
        k_fwd_chunked<NT><<<(unsigned)B, NT, smem, st>>>(status, cons, dd, start_vel, end_vel, RS, n_samples, rec, E_cap,
                                                           max_accels, bidx, bval, n_ev, vr_idx, vr_val, st_idx, n_vr, vel_f,
                                                           rounds, warm, max_rounds, ring_off);
    } else {
        if (smem > 48 * 1024) e = cudaFuncSetAttribute(k_bwd_chunked<NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return set_err("vap_velocity_profile/attr", e);
        k_bwd_chunked<NT><<<(unsigned)B, NT, smem, st>>>(status, cons, dd, dt, end_vel, RS, D_cap, n_samples, rec, E_cap,
                                                           max_accels, bidx, bval, n_ev, vel_f, vel, t_est, rounds, warm,
                                                           max_rounds, statB, ring_off);
    }
    return 0;
}

// forward and backward passes (+ the forward-only mode's slot order -> sample order) over records that are already in place
static int run_passes(int64_t B, const double* cons, const int32_t* status, double dd, double dt, double start_vel,
                      double end_vel, int64_t D_cap, const int32_t* n_samples, int E_cap, const double* max_accels,
                      const int32_t* bidx, const int32_t* bval, const int32_t* n_ev, const int32_t* vr_idx,
                      const double* vr_val, const int32_t* st_idx, const int32_t* n_vr, const double* rec,
                      const double* statB, double* vel_f, double* vel, float* t_est, int32_t* rounds, int chunks, int mode,
                      cudaStream_t stream)
{
    const long long RS = vap_pass_row_slots(D_cap, chunks);
    // CTA = one path, one chunk per thread.
    const size_t VC = 3 * (size_t)E_cap + 2;
    const size_t ss = ((size_t)chunks * 4 + E_cap + VC) * sizeof(double) + (E_cap + VC) * sizeof(int);
    // warm-up steps a speculative chunk runs before its own range (tuning: VAP_CHUNK_WARM; any value gives the same bits).
    // max_rounds only ever caps the fix-up rounds in profiling builds (-DVAP_DIAG_MAXROUNDS): it breaks exactness.
    int warm = 0, max_rounds = 1 << 30;
    if (const char* ev = getenv("VAP_CHUNK_WARM")) warm = atoi(ev);
#ifdef VAP_DIAG_MAXROUNDS
    if (const char* ev = getenv("VAP_CHUNK_MAXROUNDS")) max_rounds = atoi(ev);
#endif
    if (warm < 0) warm = 0;
    auto passes = [&](bool backward) -> int {
        switch (chunks) {
#define VAP_PASS_CASE(N_) case N_: return launch_passes<N_>(B, ss, STREAM, cons, status, dd, dt, start_vel, end_vel, RS, D_cap,    \
                                              n_samples, rec, E_cap, max_accels, bidx, bval, n_ev, vr_idx, vr_val, st_idx, n_vr,  \
                                              vel_f, vel, t_est, rounds, backward, warm, max_rounds, statB);
            VAP_PASS_CASE(8) VAP_PASS_CASE(16) VAP_PASS_CASE(32) VAP_PASS_CASE(64) VAP_PASS_CASE(128) VAP_PASS_CASE(256)
#undef VAP_PASS_CASE
        }
        return 0;
    };
    if (int rc = passes(false)) return rc;
    CHECK_LAUNCH("vap_velocity_profile/fwd");
    if (mode == 1) {                 // forward velocities only: slot order -> sample order
        const unsigned tx2 = blocks_for(D_cap, 256);
        if ((long long)tx2 * B > 2147483647LL) return arg_err("vap_velocity_profile: more than 2^31 CTAs (tile the batch)");
        k_untranspose<<<tx2 * (unsigned)B, 256, 0, STREAM>>>(status, n_samples, D_cap, RS, chunks, vel_f, vel, tx2);
        CHECK_LAUNCH("vap_velocity_profile/untranspose");
        return 0;
    }
    if (int rc = passes(true)) return rc;      // writes vel in sample order itself
    CHECK_LAUNCH("vap_velocity_profile/bwd");
    return 0;
}

static int check_pass_args(const char* who, int64_t B, int64_t D_cap, int chunks)
{
    (void)B;
    if (chunks < 8 || chunks > 256 || (chunks & (chunks - 1)) != 0) { snprintf(g_err, sizeof(g_err), "%s: chunks must be a power of two in 8 .. 256", who); return -1; }
    if (D_cap > 400000000LL) { snprintf(g_err, sizeof(g_err), "%s: D_cap too large", who); return -1; }
    if (D_cap & 1) { snprintf(g_err, sizeof(g_err), "%s: D_cap must be even (the passes move 16-byte pairs)", who); return -1; }
    return 0;
}

// S3 + S4 + S5 in one call, the fast path: distance sampling fused with the pre-pass (kappa / theta stay on chip), event
// resolution, the override fix-up of the static limits, forward and backward passes.
extern "C" int vap_velocity_profile(int64_t B, int N_max, int A_max, const double* node_attr, const int32_t* node_flags,
                                    const int32_t* n_nodes, const double* ap_attr, const int32_t* ap_flags,
                                    const int32_t* n_ap, const double* cons, const int32_t* n_splines, int32_t* status,
                                    int64_t n_grid, const double* dgrid, int samples, int64_t Q_cap, const double* lut_d,
                                    const double* lut_t, const double* total_len, int spn, int64_t P_cap,
                                    const double* prop_k, const double* prop_h, const int32_t* lut_inv, double dd, double dt,
                                    double start_vel, double end_vel, int64_t D_cap, int32_t* n_samples, double* t,
                                    double* kap, double* th, int E_cap, double* max_accels, int32_t* bidx, int32_t* bval,
                                    int32_t* n_ev, int32_t* vr_idx, double* vr_val, int32_t* st_idx, int32_t* n_vr,
                                    float* ins_est, int32_t* ev_scratch, double* rec, double* statB, double* vel_f,
                                    double* vel, float* t_est, int32_t* rounds, int chunks, int mode, void* stream)
{
    if (B <= 0) return 0;
    if (E_cap < N_max + A_max + 2) return arg_err("vap_velocity_profile: E_cap < N_max + A_max + 2");
    if (check_pass_args("vap_velocity_profile", B, D_cap, chunks)) return -1;
    if ((t != nullptr) != (kap != nullptr) || (t != nullptr) != (th != nullptr))
        return arg_err("vap_velocity_profile: t, kap and th are inspection outputs: pass all three or none");
    int Am = A_max > 0 ? A_max : 1;
    EventScratch cand;
    if (cudaError_t e = event_scratch(ev_scratch, B, N_max, Am, STREAM, cand)) return set_err("vap_velocity_profile/memset", e);
    k_count_samples<<<blocks_for(B, 128), 128, 0, STREAM>>>(B, status, status, n_grid, dgrid, total_len, D_cap, n_samples);
    CHECK_LAUNCH("vap_velocity_profile/count");
    const long long RS = vap_pass_row_slots(D_cap, chunks);
    const unsigned tx = blocks_for(D_cap + 4 * chunks, 256 * SP_TILES);
    if ((long long)tx * B > 2147483647LL) return arg_err("vap_velocity_profile: more than 2^31 CTAs (tile the batch)");
    const int tc = prepass_tile_cols(chunks);
    const size_t sm = 2 * 3 * sizeof(double) * (size_t)tc * (((256 / tc) + 2) | 1);
    k_sample_prepass<<<tx * (unsigned)B, 256, sm, STREAM>>>(N_max, Am, n_nodes, n_splines, status, cons, ap_attr, n_ap, dgrid,
                                                           samples, Q_cap, lut_d, lut_t, total_len, spn, P_cap, prop_k, prop_h,
                                                           D_cap, n_samples, t, kap, th, cand.wrap, cand.nwrap, cand.apc, cand.napc,
                                                           lut_inv, chunks, RS, rec, tx);
    CHECK_LAUNCH("vap_velocity_profile/sample_prepass");
    k_resolve_events<<<blocks_for(B, 64), 64, 0, STREAM>>>(B, N_max, Am, node_attr, node_flags, n_nodes, ap_attr, ap_flags,
                                                          n_ap, cons, status, cand.wrap, cand.nwrap, cand.apc, cand.napc, E_cap,
                                                          max_accels, bidx, bval, n_ev, vr_idx, vr_val, st_idx, n_vr, dt, ins_est);
    CHECK_LAUNCH("vap_velocity_profile/resolve");
    k_prepass_ovr<<<(unsigned)B, 256, 0, STREAM>>>(status, cons, n_samples, chunks, RS, rec, E_cap, max_accels, bidx, bval, n_ev,
                                                  statB);
    CHECK_LAUNCH("vap_velocity_profile/prepass_ovr");
    return run_passes(B, cons, status, dd, dt, start_vel, end_vel, D_cap, n_samples, E_cap, max_accels, bidx, bval, n_ev, vr_idx,
                      vr_val, st_idx, n_vr, rec, statB, vel_f, vel, t_est, rounds, chunks, mode, STREAM);
}

// ---- v2 time-domain stage ----------------------------------------------------------------------------------------
extern "C" int vap_time_profile(int64_t B, int N_max, int A_max, const double* node_attr, const int32_t* node_flags,
                                const int32_t* n_nodes, const double* ap_attr, const int32_t* ap_flags,
                                const int32_t* n_ap, const double* cons, int32_t* status, double dt, double dd,
                                const double* seg, const int32_t* first_node, const double* param_end,
                                const int32_t* n_splines, int samples, int64_t Q_cap, const double* lut_d,
                                const double* lut_t, const double* total_len, int spn, int64_t P_cap,
                                const double* prop_k, const double* prop_h, int64_t D_cap, const int32_t* n_samples,
                                const double* vel, int64_t T_cap, double* out, int32_t* nodes_map,
                                int32_t* actions_map, int32_t* n_maps, int32_t* n_out, double* summary,
                                int32_t* n_main, double* stage, int E_cap, int32_t* seg_tab, int32_t* ev_scratch,
                                int64_t out_plane_stride, const int32_t* lut_inv, const double* rden, int64_t n_rden,
                                void* stream)
{
    const long long oplane = out_plane_stride > 0 ? out_plane_stride : B * T_cap;
    if (B <= 0) return 0;
    if (E_cap < N_max + A_max + 2) return arg_err("vap_time_profile: E_cap < N_max + A_max + 2");
    int Am = A_max > 0 ? A_max : 1;
    const int64_t M_cap = T_cap;
    int32_t* seg_k = seg_tab;
    int32_t* seg_off = seg_k + (size_t)B * E_cap;
    int32_t* seg_rev = seg_off + (size_t)B * E_cap;
    int32_t* n_seg = seg_rev + (size_t)B * E_cap;
    EventScratch cand;
    if (cudaError_t e = event_scratch(ev_scratch, B, N_max, Am, STREAM, cand)) return set_err("vap_time_profile/memset", e);
    if (D_cap % 128 != 0) return arg_err("vap_time_profile: D_cap must be a multiple of 128 (rows are staged in 128-sample blocks)");
    // Serial per-path chains are latency-bound (about 4.6 cycles per dependent instruction, measured): spread the paths
    // over the warp schedulers (148 SMs x 4) with few paths per warp, so that one path's data-dependent branches stall
    // few other paths and the schedulers still have another warp to issue from.  VAP_STATE_LANES overrides (tuning).
    // More than ten paths per warp loses more to the paths' unequal lengths and block changes than a second or third warp
    // per scheduler costs (measured, 16 384 x 8 nodes: 28 lanes 6.2 ms, 10 lanes 3.8 ms for the whole time stage).
    int lanes = (int)((B + 591) / 592);
    if (lanes > 10) lanes = 10;
    if (const char* ev = getenv("VAP_STATE_LANES")) lanes = atoi(ev);
    lanes = lanes < 1 ? 1 : (lanes > 32 ? 32 : lanes);
    // ring blocks of 128 samples while every path's ring fits on the chip at once (148 SMs x 32 paths), 64 beyond
    bool big = B > 148 * 32;
    if (const char* ev = getenv("VAP_STATE_BLK")) big = atoi(ev) == 64;               // tests / tuning
    const size_t ring_bytes = (size_t)lanes * ((big ? ts_stride(64) : ts_stride(128)) * sizeof(double) + 16);   // rings + two mbarriers per path
    if (ring_bytes > 48 * 1024) {      // per device and cheap: no process-global "already set" flag (the library keeps no state)
        const int mx = (int)(32 * (ts_stride(128) * sizeof(double) + 16));
        cudaError_t ea = big ? cudaFuncSetAttribute(k_time_state<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx)
                             : cudaFuncSetAttribute(k_time_state<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx);
        if (ea != cudaSuccess) return set_err("vap_time_profile/attr", ea);
    }
    if (big)
        k_time_state<64><<<blocks_for(B, lanes), lanes, ring_bytes, STREAM>>>(B, cons, status, dt, dd, total_len, D_cap, n_samples,
                                                                             vel, M_cap, stage, n_main, rden, rden ? n_rden : 0);
    else
        k_time_state<128><<<blocks_for(B, lanes), lanes, ring_bytes, STREAM>>>(B, cons, status, dt, dd, total_len, D_cap, n_samples,
                                                                              vel, M_cap, stage, n_main, rden, rden ? n_rden : 0);
    CHECK_LAUNCH("vap_time_profile/state");
    const unsigned tx = blocks_for(M_cap, 256);
    if ((long long)tx * B > 2147483647LL) return arg_err("vap_time_profile: more than 2^31 CTAs (tile the batch)");
    const unsigned grid = tx * (unsigned)B;
    k_time_sample<<<grid, 256, 0, STREAM>>>(B, N_max, Am, n_nodes, status, ap_attr, n_ap, seg, first_node, param_end,
                                            n_splines, samples, Q_cap, lut_d, lut_t, total_len, spn, P_cap, prop_k, prop_h,
                                            M_cap, n_main, stage, cand.wrap, cand.nwrap, cand.apc, cand.napc, lut_inv, tx);
    CHECK_LAUNCH("vap_time_profile/sample");
    k_time_events<<<blocks_for(B, lanes), lanes, 0, STREAM>>>(B, N_max, Am, node_attr, node_flags, n_nodes, ap_attr, n_ap, cons,
                                                       status, dt, seg, first_node, param_end, n_splines, spn, P_cap,
                                                       prop_h, total_len, M_cap, n_main, stage, cand.wrap, cand.nwrap, cand.apc,
                                                       cand.napc, E_cap, seg_k, seg_off, seg_rev, n_seg, T_cap, oplane,
                                                       out, nodes_map, actions_map, n_maps, n_out, summary);
    CHECK_LAUNCH("vap_time_profile/events");
    k_time_finalize<<<grid, 256, 0, STREAM>>>(B, status, M_cap, n_main, stage, E_cap, seg_k, seg_off, seg_rev, n_seg,
                                              T_cap, oplane, out, summary, tx);
    CHECK_LAUNCH("vap_time_profile/finalize");
    // A path whose position moves BACKWARDS in some steps (max_dec > 0.2 / dt) can cross the same action point or node
    // boundary again and again; the parallel event detection above then runs out of candidate slots and flags the path
    // ST_EVENTS.  Such paths are redone by the reference-shaped serial kernel, one thread per path, straight into the same
    // outputs (every other thread of this launch returns after one load: a few microseconds per call).
    k_resample<<<blocks_for(B, 32), 32, 0, STREAM>>>(B, N_max, A_max, node_attr, node_flags, n_nodes, ap_attr, ap_flags, n_ap,
                                                    cons, status, dt, dd, seg, first_node, param_end, n_splines, samples,
                                                    Q_cap, lut_d, lut_t, total_len, spn, P_cap, prop_k, prop_h, D_cap,
                                                    n_samples, vel, T_cap, out, nodes_map, actions_map, n_maps, n_out,
                                                    summary, oplane, ST_EVENTS);
    CHECK_LAUNCH("vap_time_profile/serial redo");
    return 0;
}

// Measurement hook: fp64 FMA peak of the device (BASELINE.md section 3 asks for a measured DFMA figure before any fp64
// utilisation is quoted).  Every thread runs 8 independent dependent-FMA chains (more than the 8.2-cycle DFMA latency needs
// at 8 warps per scheduler); flops = ctas * 256 * iters * 8 * 2.
__global__ void __launch_bounds__(256) k_bench_dfma(long long iters, double* __restrict__ out)
{
    double a[8];
#pragma unroll
    for (int k = 0; k < 8; k++) a[k] = 1.0 + 1e-9 * (double)(threadIdx.x + 37 * k);
    const double m = 0.9999999, c = 1e-7;
    for (long long i = 0; i < iters; i++) {
#pragma unroll
        for (int k = 0; k < 8; k++) a[k] = fma(a[k], m, c);
    }
    double s = 0.0;
#pragma unroll
    for (int k = 0; k < 8; k++) s += a[k];
    if (s == 123456.789) out[0] = s;          // never true: keeps the chains alive
}
extern "C" int vap_bench_dfma(int64_t ctas, int64_t iters, double* out, void* stream)
{
    if (ctas <= 0 || iters <= 0) return 0;
    k_bench_dfma<<<(unsigned)ctas, 256, 0, STREAM>>>(iters, out);
    CHECK_LAUNCH("vap_bench_dfma");
    return 0;
}

// test hook: number of numerators (out of n pseudo-random ones) for which div_const(a, b, 1/b) != a / b
extern "C" int vap_test_div_const(int64_t n, uint64_t seed, double b, uint64_t* bad, void* stream)
{
    if (n <= 0) return 0;
    k_test_div_const<<<blocks_for(n, 256), 256, 0, STREAM>>>(n, seed, b, reinterpret_cast<unsigned long long*>(bad));
    CHECK_LAUNCH("vap_test_div_const");
    return 0;
}

// test hook: number of (num, g) pairs (out of n pseudo-random ones) for which the pass's reciprocal division differs
// from the IEEE quotient.  g covers 2|dtheta| (1e-17 .. 8, random significands, zeros, all-ones significands).
__global__ void k_test_div_recip(long long n, unsigned long long seed, unsigned long long* __restrict__ bad)
{
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    auto mix = [](unsigned long long z) {
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL; z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL; return z ^ (z >> 31);
    };
    unsigned long long z1 = mix(seed + 0x9E3779B97F4A7C15ULL * (unsigned long long)(2 * i + 1));
    unsigned long long z2 = mix(seed + 0x9E3779B97F4A7C15ULL * (unsigned long long)(2 * i + 2));
    // numerator: random sign, exponent in [-110, 8), random significand; every 64th one is +-0
    int e1 = (int)((z1 >> 52) % 118) - 110 + 1023;
    unsigned long long nb = ((z1 >> 63) << 63) | ((unsigned long long)e1 << 52) | (z1 & 0x000FFFFFFFFFFFFFULL);
    if (((z1 >> 40) & 63) == 0) nb &= 0x8000000000000000ULL;
    double num = __longlong_as_double((long long)nb);
    // denominator: positive, exponent in [-57, 3); 1/32 zeros; 1/64 all-ones significands
    int e2 = (int)((z2 >> 52) % 60) - 57 + 1023;
    unsigned long long gb = ((unsigned long long)e2 << 52) | (z2 & 0x000FFFFFFFFFFFFFULL);
    if (((z2 >> 40) & 63) == 1) gb |= 0x000FFFFFFFFFFFFFULL;
    double g = __longlong_as_double((long long)gb);
    if (((z2 >> 46) & 31) == 0) g = 0.0;
    const double rc = recip_for_pass(g);
    const double q1 = accel_ang_fast(num, g, rc);
    double n2 = num, g2 = g;
    asm volatile("" : "+d"(n2), "+d"(g2));
    const double q2 = n2 / g2;
    bool same = (__double_as_longlong(q1) == __double_as_longlong(q2)) || (q1 != q1 && q2 != q2) || (q1 == 0.0 && q2 == 0.0);
    if (!same) atomicAdd(bad, 1ULL);
}
extern "C" int vap_test_div_recip(int64_t n, uint64_t seed, uint64_t* bad, void* stream)
{
    if (n <= 0) return 0;
    k_test_div_recip<<<blocks_for(n, 256), 256, 0, STREAM>>>(n, seed, reinterpret_cast<unsigned long long*>(bad));
    CHECK_LAUNCH("vap_test_div_recip");
    return 0;
}

// dense per-path packing of the output planes (optionally straight into pinned host memory)
extern "C" int vap_pack_rows(int64_t B, int64_t T_cap, int64_t out_plane_stride, const double* out, const int32_t* n_out,
                             const int32_t* status, int64_t* offsets, double* dst, void* stream)
{
    if (B <= 0) return 0;
    const long long oplane = out_plane_stride > 0 ? out_plane_stride : B * T_cap;
    k_row_offsets<<<1, 1024, 0, STREAM>>>(B, n_out, status, T_cap, reinterpret_cast<long long*>(offsets));
    CHECK_LAUNCH("vap_pack_rows/offsets");
    int ctas = 16;
    if (const char* ev = getenv("VAP_PACK_CTAS")) ctas = atoi(ev);
    if (ctas < 1) ctas = 1;
    k_pack_rows<<<ctas, 256, 0, STREAM>>>(B, n_out, status, T_cap, oplane, out, reinterpret_cast<const long long*>(offsets), dst);
    CHECK_LAUNCH("vap_pack_rows");
    return 0;
}

// numeric rows of the trajectory export, dense per path
extern "C" int vap_export_rows(int64_t B, int64_t T_cap, int64_t out_plane_stride, const double* out, const int32_t* n_out,
                               const int32_t* status, int64_t* offsets, double* dst, void* stream)
{
    if (B <= 0) return 0;
    const long long oplane = out_plane_stride > 0 ? out_plane_stride : B * T_cap;
    k_row_offsets<<<1, 1024, 0, STREAM>>>(B, n_out, status, T_cap, reinterpret_cast<long long*>(offsets));
    CHECK_LAUNCH("vap_export_rows/offsets");
    const unsigned tx = blocks_for(T_cap, 256);
    if ((long long)tx * B > 2147483647LL) return arg_err("vap_export_rows: more than 2^31 CTAs (tile the batch)");
    const unsigned grid = tx * (unsigned)B;
    k_export_rows<<<grid, 256, 0, STREAM>>>(B, n_out, status, T_cap, oplane, out, reinterpret_cast<const long long*>(offsets), dst, tx);
    CHECK_LAUNCH("vap_export_rows");
    return 0;
}

// ---- text of the export (repr(float)-exact) -------------------------------------------------------------------------
extern "C" int vap_format_doubles(int64_t n, const double* x, char* out32, int32_t* lens, void* stream)
{
    if (n <= 0) return 0;
    k_format_doubles<<<blocks_for(n, 256), 256, 0, STREAM>>>(n, x, out32, lens);
    CHECK_LAUNCH("vap_format_doubles");
    return 0;
}
extern "C" int vap_row_text_stride(void) { return VAP_ROW_STRIDE; }
// Which entries of the result lists are Python ints in the reference (one thread per path): replays where
// generate_motion_profile inserted rows -- node 0's wait (:459-476), per crossed node i = 1 .. its turn profile (K rows,
// handle_turn :487-507) then its wait (handle_wait :509-518), per fired action point its wait (:548-553) -- from the maps
// the time stage wrote.  kinds row of path b starts at offsets[b] (dense export rows) or b * T_cap (offsets == NULL).
__global__ void k_row_kinds(long long B, int N_max, int A_max, const double* __restrict__ node_attr,
                            const int* __restrict__ n_nodes, const double* __restrict__ ap_attr, const int* __restrict__ n_ap,
                            const double* __restrict__ cons, const int* __restrict__ status, double dt,
                            const int* __restrict__ nodes_map, const int* __restrict__ actions_map,
                            const int* __restrict__ n_maps, const int* __restrict__ n_out, long long T_cap,
                            const long long* __restrict__ offsets, unsigned char* __restrict__ kinds)
{
    long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B || status[b] != ST_OK) return;
    long long T = n_out[b];
    if (T > T_cap) T = T_cap;
    unsigned char* kr = kinds + (offsets ? offsets[b] : b * T_cap);
    auto mark = [&](long long r0, long long cnt, unsigned char k) {
        for (long long r = r0; r < r0 + cnt && r < T; r++) if (r >= 0) kr[r] |= k;
    };
    const double* na = node_attr + (size_t)b * N_max * NA;
    const double V = cons[b * 6 + 0], max_acc = cons[b * 6 + 1], w = cons[b * 6 + 5];
    if (na[A_WAIT] > 0) mark(0, (long long)(na[A_WAIT] / dt), RK_INSERTED | RK_OMEGA_INT | RK_POS_INT);
    else if (T > 0) kr[0] |= RK_TIME_INT;
    const int nm = n_maps[2 * b], am = n_maps[2 * b + 1];
    const int* nmap = nodes_map + (size_t)b * (N_max + 1);
    const int n = n_nodes[b];
    for (int i = 1; i < nm - 1 && i < n; i++) {              // entry 0 is the start, the last one is len(times)
        const double* a = na + (size_t)i * NA;
        long long r = nmap[i];
        if (a[A_TURN] != 0) {
            const double angle = a[A_TURN] * (VAP_PI / 180.0);
            const Trapezoid tz = trapezoid_setup(V, max_acc, fabs(angle) * w / 2, dt);
            mark(r, 1, RK_INSERTED | RK_OMEGA_INT);
            mark(r + 1, tz.K - 1, RK_INSERTED);
            r += tz.K;
        }
        if (a[A_WAIT] > 0) mark(r, (long long)(a[A_WAIT] / dt), RK_INSERTED | RK_OMEGA_INT | RK_POS_INT);
    }
    const int* amap = actions_map + (size_t)b * (A_max > 0 ? A_max : 1);
    const int A = n_ap ? n_ap[b] : 0;
    for (int j = 0; j < am && j < A; j++) {
        const double wt = ap_attr[((size_t)b * A_max + j) * APA + P_WAIT];
        if (wt > 0) mark(amap[j], (long long)(wt / dt), RK_INSERTED | RK_OMEGA_INT | RK_POS_INT);
    }
}

extern "C" int vap_row_kinds(int64_t B, int N_max, int A_max, const double* node_attr, const int32_t* n_nodes,
                             const double* ap_attr, const int32_t* n_ap, const double* cons, const int32_t* status,
                             double dt, const int32_t* nodes_map, const int32_t* actions_map, const int32_t* n_maps,
                             const int32_t* n_out, int64_t T_cap, const int64_t* offsets, int64_t n_kinds, uint8_t* kinds,
                             void* stream)
{
    if (B <= 0 || n_kinds <= 0) return 0;
    cudaError_t e = cudaMemsetAsync(kinds, 0, (size_t)n_kinds, STREAM);
    if (e != cudaSuccess) return set_err("vap_row_kinds/memset", e);
    k_row_kinds<<<blocks_for(B, 64), 64, 0, STREAM>>>(B, N_max, A_max, node_attr, n_nodes, ap_attr, n_ap, cons, status, dt,
                                                     nodes_map, actions_map, n_maps, n_out, T_cap,
                                                     reinterpret_cast<const long long*>(offsets), kinds);
    CHECK_LAUNCH("vap_row_kinds");
    return 0;
}

extern "C" int vap_format_rows(int64_t R, const double* rows, const uint8_t* int_time, char* slots, int32_t* lens, void* stream)
{
    if (R <= 0) return 0;
    k_format_rows<<<blocks_for(R, 128), 128, 0, STREAM>>>(R, rows, int_time, slots, lens);
    CHECK_LAUNCH("vap_format_rows");
    return 0;
}
extern "C" int vap_compact_rows(int64_t R, const char* slots, const int32_t* lens, const int64_t* offsets, char* text,
                                void* stream)
{
    if (R <= 0) return 0;
    k_compact_rows<<<blocks_for(R * 32, 256), 256, 0, STREAM>>>(R, slots, lens, reinterpret_cast<const long long*>(offsets), text);
    CHECK_LAUNCH("vap_compact_rows");
    return 0;
}

extern "C" int vap_splice_plan(int64_t B, int N_max, int A_max, const int32_t* status, const int32_t* nodes_map,
                               const int32_t* actions_map, const int32_t* n_maps, const int64_t* row_offsets,
                               const int64_t* line_offsets, const int64_t* act_first, const int32_t* act_rows, int64_t n_act,
                               const int64_t* act_off, int64_t* path_offsets, int64_t* line_dst, int64_t* act_dst,
                               int32_t* flags, void* stream)
{
    if (B <= 0) return 0;
    if (N_max < 1 || A_max < 0 || n_act < 0) return arg_err("vap_splice_plan: N_max >= 1, A_max >= 0 and n_act >= 0 required");
    const int A_stride = A_max > 0 ? A_max : 1;
    const size_t warp_bytes = (size_t)4 * sizeof(long long) * (size_t)(N_max + 1 + A_stride);
    int max_smem = 0, dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    if (e != cudaSuccess) return set_err("vap_splice_plan/attr", e);
    if (warp_bytes > (size_t)max_smem) return arg_err("vap_splice_plan: N_max + A_max too large for one warp's shared memory");
    int warps = 4;
    while (warps > 1 && warps * warp_bytes > 48 * 1024) warps >>= 1;
    const size_t smem = warps * warp_bytes;
    if (smem > 48 * 1024) {
        e = cudaFuncSetAttribute(k_splice_plan, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return set_err("vap_splice_plan/attr", e);
    }
    if (n_act > 0) {
        e = cudaMemsetAsync(act_dst, 0xff, (size_t)n_act * sizeof(int64_t), STREAM);     // -1: the row is in no body
        if (e != cudaSuccess) return set_err("vap_splice_plan/memset", e);
    }
    const long long* ro = reinterpret_cast<const long long*>(row_offsets);
    const long long* lo = reinterpret_cast<const long long*>(line_offsets);
    const long long* af = reinterpret_cast<const long long*>(act_first);
    const long long* ao = reinterpret_cast<const long long*>(act_off);
    long long* po = reinterpret_cast<long long*>(path_offsets);
    k_splice_offsets<<<1, 1024, 0, STREAM>>>(B, N_max, A_stride, status, n_maps, ro, lo, af, act_rows, n_act, ao, po, flags);
    CHECK_LAUNCH("vap_splice_plan/offsets");
    k_splice_plan<<<blocks_for(B, warps), warps * 32, smem, STREAM>>>(B, N_max, A_stride, nodes_map, actions_map, n_maps, ro, lo,
                                                                     af, act_rows, ao, po, flags,
                                                                     reinterpret_cast<long long*>(line_dst),
                                                                     reinterpret_cast<long long*>(act_dst));
    CHECK_LAUNCH("vap_splice_plan");
    return 0;
}

extern "C" int vap_splice_actions(int64_t n_act, const char* act_text, const int64_t* act_off, const int64_t* act_dst,
                                  char* text, void* stream)
{
    if (n_act <= 0) return 0;
    k_splice_actions<<<blocks_for(n_act * 32, 256), 256, 0, STREAM>>>(n_act, act_text, reinterpret_cast<const long long*>(act_off),
                                                                     reinterpret_cast<const long long*>(act_dst), text);
    CHECK_LAUNCH("vap_splice_actions");
    return 0;
}

// ---- reading the text back (vap_parse.cuh) ------------------------------------------------------------------------
extern "C" int vap_parse_doubles(int64_t n, const char* text, const int64_t* tok_off, double* out, int8_t* flags, void* stream)
{
    if (n <= 0) return 0;
    k_parse_doubles<<<blocks_for(n, 256), 256, 0, STREAM>>>(n, text, reinterpret_cast<const long long*>(tok_off), out,
                                                           reinterpret_cast<signed char*>(flags));
    CHECK_LAUNCH("vap_parse_doubles");
    return 0;
}

extern "C" int vap_line_starts(int64_t B, int64_t n_bytes, const char* text, const int64_t* path_off, uint8_t* starts,
                               void* stream)
{
    if (B < 0 || n_bytes < 0) return arg_err("vap_line_starts: B >= 0 and n_bytes >= 0 required");
    if (n_bytes == 0) return 0;
    k_line_starts<<<blocks_for(n_bytes, 256), 256, 0, STREAM>>>(n_bytes, text, starts);
    CHECK_LAUNCH("vap_line_starts");
    if (B > 0) {
        k_body_starts<<<blocks_for(B, 256), 256, 0, STREAM>>>(B, n_bytes, reinterpret_cast<const long long*>(path_off), starts);
        CHECK_LAUNCH("vap_line_starts/bodies");
    }
    return 0;
}

extern "C" int vap_line_offsets(int64_t B, int64_t n_bytes, const uint8_t* starts, const int32_t* scan, const int64_t* path_off,
                                int64_t* line_off, int64_t* path_line_off, void* stream)
{
    if (B < 0 || n_bytes < 0) return arg_err("vap_line_offsets: B >= 0 and n_bytes >= 0 required");
    if (n_bytes > 0) {
        k_line_offsets<<<blocks_for(n_bytes, 256), 256, 0, STREAM>>>(n_bytes, starts, scan, reinterpret_cast<long long*>(line_off));
        CHECK_LAUNCH("vap_line_offsets");
    }
    k_path_lines<<<blocks_for(B + 1, 256), 256, 0, STREAM>>>(B, n_bytes, reinterpret_cast<const long long*>(path_off), scan,
                                                            reinterpret_cast<long long*>(line_off),
                                                            reinterpret_cast<long long*>(path_line_off));
    CHECK_LAUNCH("vap_line_offsets/paths");
    return 0;
}

extern "C" int vap_line_kinds(int64_t L, const char* text, const int64_t* line_off, uint8_t* kinds, int32_t* errors,
                              int64_t* counts, void* stream)
{
    if (L <= 0) return 0;
    if (L >= (1LL << 31)) return arg_err("vap_line_kinds: at most 2^31 - 1 lines");
    k_line_kinds<<<blocks_for(L, 256), 256, 0, STREAM>>>(L, text, reinterpret_cast<const long long*>(line_off), kinds, errors,
                                                        reinterpret_cast<long long*>(counts));
    CHECK_LAUNCH("vap_line_kinds");
    return 0;
}

extern "C" int vap_parse_rows(int64_t B, int64_t L, const char* text, const int64_t* line_off, const uint8_t* kinds,
                              const int64_t* count_scan, const int64_t* path_line_off, int64_t parse_paths,
                              int64_t* path_row_off, int64_t* path_act_off, int64_t* act_line, double* rows,
                              uint8_t* host_mask, int32_t* errors, void* stream)
{
    if (B < 0 || L < 0 || parse_paths < 0 || parse_paths > B)
        return arg_err("vap_parse_rows: B >= 0, L >= 0 and 0 <= parse_paths <= B required");
    const long long* cs = reinterpret_cast<const long long*>(count_scan);
    const long long* pl = reinterpret_cast<const long long*>(path_line_off);
    k_path_rows<<<blocks_for(B + 1, 256), 256, 0, STREAM>>>(B, pl, cs, reinterpret_cast<long long*>(path_row_off),
                                                           reinterpret_cast<long long*>(path_act_off));
    CHECK_LAUNCH("vap_parse_rows/paths");
    if (L == 0) return 0;
    cudaError_t e = cudaMemsetAsync(host_mask, 0, (size_t)L, STREAM);
    if (e != cudaSuccess) return set_err("vap_parse_rows/memset", e);
    k_parse_lines<<<blocks_for(L, 128), 128, 0, STREAM>>>(L, text, reinterpret_cast<const long long*>(line_off), kinds, cs,
                                                         pl + parse_paths, reinterpret_cast<long long*>(act_line), rows,
                                                         host_mask, errors);
    CHECK_LAUNCH("vap_parse_rows");
    return 0;
}

extern "C" int vap_compare_bodies(int64_t B, const char* text, const int64_t* old_off, const int64_t* new_off,
                                  const int64_t* line_off, const int32_t* line_err, const int64_t* old_path_line_off,
                                  const int64_t* act_line, const int64_t* old_path_act_off, const int64_t* new_path_act_off,
                                  const double* old_rows, const int64_t* old_row_off, const double* new_rows,
                                  const int64_t* new_row_off, int64_t* out_i64, double* out_f64, void* stream)
{
    if (B <= 0) return 0;
    typedef const long long* P;
    k_compare_bodies<<<blocks_for(B * 32, 128), 128, 0, STREAM>>>(B, text, P(old_off), P(new_off), P(line_off), line_err,
                                                                  P(old_path_line_off), P(act_line), P(old_path_act_off),
                                                                  P(new_path_act_off), old_rows, P(old_row_off), new_rows,
                                                                  P(new_row_off), reinterpret_cast<long long*>(out_i64), out_f64);
    CHECK_LAUNCH("vap_compare_bodies");
    return 0;
}

// ---- the robot's footprint along the export rows (vap_footprint.cuh) ------------------------------------------------
extern "C" int vap_footprint_check(int64_t B, const double* rows, const int64_t* row_off, double hl, double hw, double xmin,
                                   double xmax, double ymin, double ymax, int K, const double* boxes, double tol,
                                   int64_t* out_i64, double* out_f64, void* stream)
{
    if (B < 0) return arg_err("vap_footprint_check: B >= 0 required");
    if (!(hl > 0) || !(hw > 0) || !isfinite(hl) || !isfinite(hw))
        return arg_err("vap_footprint_check: the half-length and half-width must be positive and finite");
    if (!(xmin < xmax) || !(ymin < ymax)) return arg_err("vap_footprint_check: empty field box (xmin < xmax and ymin < ymax required)");
    if (!isfinite(tol)) return arg_err("vap_footprint_check: the tolerance must be finite");
    if (K < 0 || K > FP_MAX_BOXES) return arg_err("vap_footprint_check: 0 <= K <= 64 keep-out boxes required");
    if (K > 0 && boxes == nullptr) return arg_err("vap_footprint_check: boxes is NULL");
    FpArgs a;
    memset(&a, 0, sizeof(a));
    a.hl = hl; a.hw = hw; a.xmin = xmin; a.xmax = xmax; a.ymin = ymin; a.ymax = ymax; a.tol = tol; a.K = K;
    for (int k = 0; k < K; k++) {
        const double* q = boxes + 4 * k;
        if (!(q[0] < q[2]) || !(q[1] < q[3]) || !isfinite(q[0]) || !isfinite(q[1]) || !isfinite(q[2]) || !isfinite(q[3])) {
            snprintf(g_err, sizeof(g_err), "vap_footprint_check: keep-out box %d is empty or not finite (x0 < x1 and y0 < y1 "
                     "required, got %g, %g, %g, %g)", k, q[0], q[1], q[2], q[3]);
            return -101;
        }
        for (int j = 0; j < 4; j++) a.box[k][j] = q[j];
    }
    if (B == 0) return 0;
    const unsigned grid = (unsigned)(B < 1048576 ? B : 1048576);
    k_footprint_check<<<grid, FP_THREADS, 0, STREAM>>>(B, rows, reinterpret_cast<const long long*>(row_off), a,
                                                       reinterpret_cast<long long*>(out_i64), out_f64);
    CHECK_LAUNCH("vap_footprint_check");
    return 0;
}

// =====================================================================================================
// The whole hot path behind ONE call (SURVEY.md 8b): generate_motion_profile(spline_manager, constraints)
// (motion_profile_generator.py:389-628, incl. build_path and rebuild_tables) for a batch, out of one caller workspace.
// =====================================================================================================
#define VAP_DIST_LIMIT 5.0e7     // more distance samples than this per path (an infinite length too): ST_DIVERGED
#define VAP_TIME_LIMIT 1.0e7     // more time samples than this per path: treated as a non-terminating profile (ST_DIVERGED)

// paths whose sampling loop `while d < total_length` would never end / never fit are flagged before anything is sized on them
__global__ void k_flag_lengths(long long B, const int* __restrict__ gstatus, const double* __restrict__ total_len, double dd,
                               int* __restrict__ status)
{
    long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    int s = gstatus[b];
    if (s == ST_OK && total_len[b] / dd > VAP_DIST_LIMIT) s = ST_DIVERGED;      // false for NaN (the reference's loops do not run)
    status[b] = s;
}
// after the velocity stage: flag absurd travel times, publish what the batch needs (need[0] = max distance samples,
// need[1] = max estimated time samples incl. inserted rows; both over healthy paths) so that a caller can size a retry
__global__ void k_flag_times(long long B, int* __restrict__ status, const int* __restrict__ n_samples,
                             const float* __restrict__ t_est, const float* __restrict__ ins_est,
                             unsigned long long* __restrict__ need)
{
    long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const int s = status[b];
    if (s != ST_OK && s != ST_CAPACITY) return;
    atomicMax(need, (unsigned long long)(n_samples[b] > 0 ? n_samples[b] : 0));
    if (s != ST_OK) return;
    const float est = t_est[b] + ins_est[b];
    if (!(est < (float)VAP_TIME_LIMIT)) { status[b] = ST_DIVERGED; return; }
    atomicMax(need + 1, (unsigned long long)est);
}
// row counts once the time stage has run: the main-loop iterations (exact even when the rows did not fit) plus the bound of
// the rows that waits and turn profiles insert
__global__ void k_need_rows(long long B, const int* __restrict__ status, const int* __restrict__ n_main,
                            const float* __restrict__ ins_est, unsigned long long* __restrict__ need)
{
    long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const int s = status[b];
    if (s == ST_OK || s == ST_CAPACITY)
        atomicMax(need + 2, (unsigned long long)(n_main[b] > 0 ? n_main[b] : 0) + (unsigned long long)ceilf(ins_est[b]) + 8ull);
}

struct WsCarver {
    char* base; size_t off;
    template <typename T> T* take(size_t n)
    {
        off = (off + 255) & ~(size_t)255;
        T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
        off += n * sizeof(T);
        return p;
    }
};
struct BatchScratch {
    double *seg, *param_end, *seglen, *scratch9, *lut_d, *lut_t, *total_len, *prop_k, *prop_h, *ma, *vr_val, *rec, *statB, *vel_f,
           *stage;
    int32_t *first_node, *n_splines, *gstatus, *lut_inv, *bidx, *bval, *n_ev, *vr_idx, *st_idx, *n_vr, *scr, *rounds, *seg_tab,
            *scr2, *n_main;
    float *ins_est, *t_est;
    unsigned long long* need;
    int64_t Q_cap, P_cap, RS; int E_cap;
};
static size_t carve_batch(char* base, int64_t B, int N_max, int A_max, int max_splines, int samples, int spn, int64_t D_cap,
                          int64_t T_cap, int chunks, BatchScratch& s)
{
    WsCarver w{base, 0};
    const int S = max_splines > 0 ? max_splines : 1;
    s.Q_cap = (int64_t)samples * S; s.P_cap = (int64_t)spn * N_max; s.E_cap = N_max + A_max + 2;
    s.RS = vap_pass_row_slots(D_cap, chunks);
    const size_t nscr = (size_t)vap_event_scratch_ints(B, N_max, A_max);
    s.seg = w.take<double>((size_t)B * (N_max > 1 ? N_max - 1 : 1) * 12);
    s.first_node = w.take<int32_t>((size_t)B * (N_max + 1));
    s.param_end = w.take<double>((size_t)B * N_max);
    s.seglen = w.take<double>((size_t)B * N_max);
    s.n_splines = w.take<int32_t>(B);
    s.gstatus = w.take<int32_t>(B);
    s.scratch9 = w.take<double>((size_t)B * N_max * 9);
    s.lut_d = w.take<double>((size_t)B * s.Q_cap);
    s.lut_t = w.take<double>((size_t)B * s.Q_cap);
    s.total_len = w.take<double>(B);
    s.lut_inv = w.take<int32_t>((size_t)B * vap_lut_index_row_ints(s.Q_cap));
    s.prop_k = w.take<double>((size_t)B * s.P_cap);
    s.prop_h = w.take<double>((size_t)B * s.P_cap);
    s.ma = w.take<double>((size_t)B * s.E_cap);
    s.bidx = w.take<int32_t>((size_t)B * s.E_cap);
    s.bval = w.take<int32_t>((size_t)B * s.E_cap);
    s.n_ev = w.take<int32_t>((size_t)B * 2);
    s.vr_idx = w.take<int32_t>((size_t)B * s.E_cap);
    s.vr_val = w.take<double>((size_t)B * s.E_cap);
    s.st_idx = w.take<int32_t>((size_t)B * s.E_cap);
    s.n_vr = w.take<int32_t>((size_t)B * 2);
    s.ins_est = w.take<float>(B);
    s.t_est = w.take<float>(B);
    s.scr = w.take<int32_t>(nscr);
    s.rounds = w.take<int32_t>((size_t)B * 2);
    s.rec = w.take<double>((size_t)B * s.RS * 4);
    s.statB = w.take<double>((size_t)B * s.RS);
    s.vel_f = w.take<double>((size_t)B * s.RS);
    s.stage = w.take<double>((size_t)8 * B * (T_cap + 1));
    s.seg_tab = w.take<int32_t>((size_t)3 * B * s.E_cap + B);
    s.scr2 = w.take<int32_t>(nscr);
    s.n_main = w.take<int32_t>(B);
    s.need = w.take<unsigned long long>(4);
    return (w.off + 255) & ~(size_t)255;
}

static int check_batch_args(const char* who, int64_t B, int N_max, int A_max, int max_splines, int samples, int spn,
                            int64_t D_cap, int64_t T_cap, int chunks)
{
    if (B < 0 || N_max < 2 || A_max < 0 || max_splines < 1 || max_splines > N_max || samples < 2 || spn < 2 || T_cap < 1) {
        snprintf(g_err, sizeof(g_err), "%s: bad sizes", who); return -1;
    }
    if (D_cap < 128 || D_cap % 128 != 0) { snprintf(g_err, sizeof(g_err), "%s: D_cap must be a positive multiple of 128", who); return -1; }
    return check_pass_args(who, B, D_cap, chunks);
}

extern "C" int64_t vap_workspace_bytes(int64_t B, int N_max, int A_max, int max_splines, int lut_samples, int samples_per_node,
                                       int64_t D_cap, int64_t T_cap, int chunks)
{
    if (check_batch_args("vap_workspace_bytes", B, N_max, A_max, max_splines, lut_samples, samples_per_node, D_cap, T_cap, chunks))
        return -1;
    BatchScratch s;
    return (int64_t)carve_batch(nullptr, B, N_max, A_max, max_splines, lut_samples, samples_per_node, D_cap, T_cap, chunks, s);
}

extern "C" int vap_profile_batch(int64_t B, int N_max, int A_max, int max_splines, const double* node_attr,
                                 const int32_t* node_flags, const int32_t* n_nodes, const double* ap_attr,
                                 const int32_t* ap_flags, const int32_t* n_ap, const double* cons, double dt, double dd,
                                 double start_vel, double end_vel, int lut_samples, int samples_per_node, int64_t D_cap,
                                 int64_t T_cap, int chunks, const double* dgrid, int64_t n_grid, const double* rden,
                                 int64_t n_rden, void* workspace, int64_t workspace_bytes, double* out,
                                 int64_t out_plane_stride, int32_t* n_out, int32_t* nodes_map, int32_t* actions_map,
                                 int32_t* n_maps, int32_t* status, double* summary, double* vel, int32_t* n_samples,
                                 int64_t* need, void* stream)
{
    if (B == 0) return 0;
    if (check_batch_args("vap_profile_batch", B, N_max, A_max, max_splines, lut_samples, samples_per_node, D_cap, T_cap, chunks))
        return -1;
    if (!dgrid || n_grid < D_cap + 2) return arg_err("vap_profile_batch: dgrid (vap_build_dgrid) must hold at least D_cap + 2 entries");
    if (!workspace) return arg_err("vap_profile_batch: workspace is NULL");
    BatchScratch s;
    const size_t bytes = carve_batch(static_cast<char*>(workspace), B, N_max, A_max, max_splines, lut_samples, samples_per_node,
                                     D_cap, T_cap, chunks, s);
    if ((int64_t)bytes > workspace_bytes) return arg_err("vap_profile_batch: workspace smaller than vap_workspace_bytes(...)");
    if ((reinterpret_cast<uintptr_t>(workspace) & 255) != 0) return arg_err("vap_profile_batch: workspace must be 256-byte aligned");
    cudaError_t e = cudaMemsetAsync(s.need, 0, 4 * sizeof(unsigned long long), STREAM);
    if (e != cudaSuccess) return set_err("vap_profile_batch/memset", e);
    int rc;
    // S0 build_path, S1 distance table (+ inverse index), S2 curvature / heading tables  (rebuild_tables, spline_manager.py:582)
    if ((rc = vap_build_path(B, N_max, node_attr, node_flags, n_nodes, s.seg, s.first_node, s.param_end, s.seglen, s.n_splines,
                             s.gstatus, s.scratch9, nullptr, nullptr, stream))) return rc;
    if ((rc = vap_build_lut(B, N_max, s.seg, s.first_node, s.param_end, s.n_splines, s.gstatus, lut_samples, s.Q_cap, s.lut_d,
                            s.lut_t, s.total_len, stream))) return rc;
    if ((rc = vap_build_lut_index(B, s.n_splines, s.gstatus, lut_samples, s.Q_cap, s.lut_d, s.total_len, s.lut_inv, stream))) return rc;
    if ((rc = vap_build_props(B, N_max, n_nodes, s.seg, s.first_node, s.param_end, s.n_splines, s.gstatus, samples_per_node,
                              s.P_cap, s.prop_k, s.prop_h, stream))) return rc;
    k_flag_lengths<<<blocks_for(B, 128), 128, 0, STREAM>>>(B, s.gstatus, s.total_len, dd, status);
    CHECK_LAUNCH("vap_profile_batch/flag_lengths");
    // S3 + S4 + S5
    if ((rc = vap_velocity_profile(B, N_max, A_max, node_attr, node_flags, n_nodes, ap_attr, ap_flags, n_ap, cons, s.n_splines,
                                   status, n_grid, dgrid, lut_samples, s.Q_cap, s.lut_d, s.lut_t, s.total_len, samples_per_node,
                                   s.P_cap, s.prop_k, s.prop_h, s.lut_inv, dd, dt, start_vel, end_vel, D_cap, n_samples, nullptr,
                                   nullptr, nullptr, s.E_cap, s.ma, s.bidx, s.bval, s.n_ev, s.vr_idx, s.vr_val, s.st_idx, s.n_vr,
                                   s.ins_est, s.scr, s.rec, s.statB, s.vel_f, vel, s.t_est, s.rounds, chunks, 0, stream))) return rc;
    k_flag_times<<<blocks_for(B, 128), 128, 0, STREAM>>>(B, status, n_samples, s.t_est, s.ins_est, s.need);
    CHECK_LAUNCH("vap_profile_batch/flag_times");
    // S6 + S7
    if ((rc = vap_time_profile(B, N_max, A_max, node_attr, node_flags, n_nodes, ap_attr, ap_flags, n_ap, cons, status, dt, dd,
                               s.seg, s.first_node, s.param_end, s.n_splines, lut_samples, s.Q_cap, s.lut_d, s.lut_t, s.total_len,
                               samples_per_node, s.P_cap, s.prop_k, s.prop_h, D_cap, n_samples, vel, T_cap, out, nodes_map,
                               actions_map, n_maps, n_out, summary, s.n_main, s.stage, s.E_cap, s.seg_tab, s.scr2,
                               out_plane_stride, s.lut_inv, rden, rden ? n_rden : 0, stream))) return rc;
    k_need_rows<<<blocks_for(B, 128), 128, 0, STREAM>>>(B, status, s.n_main, s.ins_est, s.need);
    CHECK_LAUNCH("vap_profile_batch/need_rows");
    if (need) {
        e = cudaMemcpyAsync(need, s.need, 3 * sizeof(int64_t), cudaMemcpyDeviceToDevice, STREAM);
        if (e != cudaSuccess) return set_err("vap_profile_batch/need", e);
    }
    return 0;
}

// S7 on its own: summary[b] = {n_out, total_length, times[-1], max |linear_vels|, status} from the output streams
// (what the ranks of a sharded job gather; vap_resample / vap_time_profile / vap_profile_batch already write it).
__global__ void __launch_bounds__(128) k_summary(long long T_cap, long long plane, const double* __restrict__ out,
                                                 const int* __restrict__ n_out, const int* __restrict__ status,
                                                 const double* __restrict__ total_len, double* __restrict__ summary)
{
    const long long b = blockIdx.x;
    __shared__ double s_m[128];
    const int st = status[b];
    const long long T = (st == ST_OK) ? n_out[b] : 0;
    const double* v = out + 2 * plane + (size_t)b * T_cap;
    double m = 0.0;
    for (long long i = threadIdx.x; i < T; i += blockDim.x) m = fmax(m, fabs(v[i]));
    s_m[threadIdx.x] = m;
    __syncthreads();
    for (int k = 64; k > 0; k >>= 1) { if ((int)threadIdx.x < k) s_m[threadIdx.x] = fmax(s_m[threadIdx.x], s_m[threadIdx.x + k]); __syncthreads(); }
    if (threadIdx.x == 0) {
        double* r = summary + (size_t)b * 5;
        r[0] = (double)n_out[b]; r[1] = total_len ? total_len[b] : 0.0;
        r[2] = T > 0 ? out[(size_t)b * T_cap + T - 1] : 0.0; r[3] = s_m[0]; r[4] = (double)st;
    }
}
extern "C" int vap_summary(int64_t B, int64_t T_cap, int64_t out_plane_stride, const double* out, const int32_t* n_out,
                           const int32_t* status, const double* total_len, double* summary, void* stream)
{
    if (B <= 0) return 0;
    const long long plane = out_plane_stride > 0 ? out_plane_stride : B * T_cap;
    k_summary<<<(unsigned)B, 128, 0, STREAM>>>(T_cap, plane, out, n_out, status, total_len, summary);
    CHECK_LAUNCH("vap_summary");
    return 0;
}

// bounds diagnostics (see vap_device.cuh): out[32] = violations per site (0..15) and checks executed per site (16..31);
// returns -1 in a build without -DVAP_BOUNDS_CHECK.  reset != 0 clears the counters afterwards.
extern "C" int vap_diag_read(uint64_t* out_host, int reset)
{
#ifdef VAP_BOUNDS_CHECK
    cudaError_t e = cudaMemcpyFromSymbol(out_host, g_vap_diag, sizeof(unsigned long long) * VAP_DIAG_SITES);
    if (e != cudaSuccess) return set_err("vap_diag_read", e);
    if (reset) {
        unsigned long long z[VAP_DIAG_SITES] = {0};
        e = cudaMemcpyToSymbol(g_vap_diag, z, sizeof(z));
        if (e != cudaSuccess) return set_err("vap_diag_read/reset", e);
    }
    return 0;
#else
    (void)out_host; (void)reset;
    return arg_err("vap_diag_read: this build has no bounds diagnostics (compile with -DVAP_BOUNDS_CHECK)");
#endif
}
