// vap_velocity.cuh -- stages S3-events / S4 / S5: sample-parallel event detection, a pre-pass that hoists every term of
// the forward / backward recurrences that depends neither on the velocity state nor on the events into four values per
// sample (chunk-interleaved rows, written once), and chunk-speculative kernels that run the exact serial recurrences on
// many chunks of one path at once over coalesced streams.
//
// Exactness: the recurrences of motion_profile_generator.py:188-311 are NOT associative (the wheel-acceleration
// term depends on v[i] and v[i-1], SURVEY.md F4), so no scan is used.  A chunk starts from a guessed state, and
// is re-run from its predecessor's true end state until two consecutive velocities are BITWISE equal to the ones
// computed before; from there on the old results are the serial results.  The fix-up loop ends when no chunk
// changed, at which point (by induction from chunk 0) every value equals the serial evaluation bit for bit.
#pragma once
#include "vap_device.cuh"

#define EV_AP_CAND 4

// read-only (ld.global.nc) load of a 32-byte record
__device__ __forceinline__ double4 ldg_d4(const double4* p)
{
    const double2* q = reinterpret_cast<const double2*>(p);
    double2 a = __ldg(q), b = __ldg(q + 1);
    return make_double4(a.x, a.y, b.x, b.y);
}

// ---- S3 (per path): replay the sampling loop's event logic over the candidate samples only --------------------
// Outputs the reference's max_accels / boundary_map plus the piecewise-constant initial-velocity regimes:
//   vr_idx/vr_val: v0[i] = vr_val[j] for the last j with vr_idx[j] <= i      (max_velocity before sample i's events)
//   st_idx       : samples whose initial velocity is overwritten with 0.01    (stop nodes / stop action points)
__global__ void k_resolve_events(long long B, int N_max, int A_max, const double* __restrict__ node_attr,
                                 const int* __restrict__ node_flags, const int* __restrict__ n_nodes,
                                 const double* __restrict__ ap_attr, const int* __restrict__ ap_flags,
                                 const int* __restrict__ n_ap, const double* __restrict__ cons,
                                 int* __restrict__ status, int* __restrict__ ev_wrap, const int* __restrict__ ev_nwrap,
                                 const int* __restrict__ ev_apc, const int* __restrict__ ev_napc, int E_cap,
                                 double* __restrict__ max_accels, int* __restrict__ bidx, int* __restrict__ bval,
                                 int* __restrict__ n_ev, int* __restrict__ vr_idx, double* __restrict__ vr_val,
                                 int* __restrict__ st_idx, int* __restrict__ n_vr, double dt,
                                 float* __restrict__ ins_est)
{
    long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    n_ev[2 * b] = 0; n_ev[2 * b + 1] = 0; n_vr[2 * b] = 0; n_vr[2 * b + 1] = 0;
    if (ins_est) ins_est[b] = 0.f;
    if (status[b] != ST_OK) return;
    const int n = n_nodes[b];
    const int A = n_ap ? n_ap[b] : 0;
    const double* na = node_attr + (size_t)b * N_max * NA;
    const int* nf = node_flags + (size_t)b * N_max;
    const double* apa = ap_attr + (size_t)b * A_max * APA;
    const int* apf = ap_flags + (size_t)b * A_max;
    const double V = cons[b * 6 + 0], A0 = cons[b * 6 + 1];
    double* ma = max_accels + (size_t)b * E_cap;
    int* bi = bidx + (size_t)b * E_cap;
    int* bv = bval + (size_t)b * E_cap;
    int* vi = vr_idx + (size_t)b * E_cap;
    double* vv = vr_val + (size_t)b * E_cap;
    int* si = st_idx + (size_t)b * E_cap;
    int* wr = ev_wrap + (size_t)b * N_max;
    int nw = ev_nwrap[b];
    if (nw > N_max) { status[b] = ST_EVENTS; return; }
    // sort the wrap samples ascending: they arrive in the order of the atomics, i.e. by tile of the chunk-interleaved
    // sampling kernel (far from sorted), so a shell sort (Ciura gaps) instead of a plain insertion sort: a path with 800 nodes
    // took 6.9 ms here with the latter
    {
        const int gaps[9] = {1750, 701, 301, 132, 57, 23, 10, 4, 1};
        for (int gi = 0; gi < 9; gi++) {
            const int gap = gaps[gi];
            if (gap >= nw) continue;
            for (int i = gap; i < nw; i++) {
                const int x = wr[i];
                int j = i - gap;
                while (j >= 0 && wr[j] > x) { wr[j + gap] = wr[j]; j -= gap; }
                wr[j + gap] = x;
            }
        }
    }
    int n_acc = 0, n_b = 0, nvr = 0, nst = 0;
    double max_velocity = (na[A_MAXVEL] > 0) ? na[A_MAXVEL] : V;
    ma[n_acc++] = (na[A_MAXACC] > 0) ? na[A_MAXACC] : A0;
    bi[0] = 0; bv[0] = 0; n_b = 1;
    vi[nvr] = 0; vv[nvr] = max_velocity; nvr++;
    // action point k fires at its smallest candidate sample after the previous action point's sample
    int node_num = 0, wptr = 0, action_idx = 0, last_fire = -1;
    bool actions_dead = false;
    while (true) {
        // next action-point sample (if any)
        int ai = 2147483647;
        if (!actions_dead && action_idx < A) {
            int nc = ev_napc[(size_t)b * A_max + action_idx];
            if (nc > EV_AP_CAND) { status[b] = ST_EVENTS; return; }
            const int* c = ev_apc + ((size_t)b * A_max + action_idx) * EV_AP_CAND;
            for (int k = 0; k < nc; k++) if (c[k] > last_fire && c[k] < ai) ai = c[k];
            if (ai == 2147483647) actions_dead = true;      // this action point never fires -> none after it does
        }
        int wi = (wptr < nw) ? wr[wptr] : 2147483647;
        if (wi == 2147483647 && ai == 2147483647) break;
        int i = wi < ai ? wi : ai;
        bool stop = false;
        if (wi == i) {                       // node crossing first (:124-140)
            wptr++;
            node_num += 1;
            const double* a = na + (size_t)node_num * NA;
            if (nf[node_num] & F_STOP) stop = true;
            max_velocity = (a[A_MAXVEL] > 0) ? a[A_MAXVEL] : V;
            ma[n_acc++] = (a[A_MAXACC] > 0) ? a[A_MAXACC] : A0;
            if (node_num < n - 1) {
                if (bi[n_b - 1] == i) bv[n_b - 1] = n_acc - 1;
                else { bi[n_b] = i; bv[n_b] = n_acc - 1; n_b++; }
            }
        }
        if (ai == i) {                       // then the action point (:142-163)
            const double* p = apa + (size_t)action_idx * APA;
            max_velocity = (p[P_MAXVEL] > 0) ? p[P_MAXVEL] : V;
            if (apf[action_idx] & F_STOP) stop = true;
            ma[n_acc++] = (p[P_MAXACC] > 0) ? p[P_MAXACC] : A0;
            if (bi[n_b - 1] == i) bv[n_b - 1] = n_acc - 1;
            else { bi[n_b] = i; bv[n_b] = n_acc - 1; n_b++; }
            action_idx += 1;
            last_fire = i;
        }
        if (stop) si[nst++] = i;
        if (vi[nvr - 1] == i + 1) vv[nvr - 1] = max_velocity;
        else { vi[nvr] = i + 1; vv[nvr] = max_velocity; nvr++; }
    }
    ma[n_acc++] = A0;
    n_ev[2 * b] = n_acc; n_ev[2 * b + 1] = n_b;
    n_vr[2 * b] = nvr; n_vr[2 * b + 1] = nst;
    if (ins_est) {
        // rows the time-domain stage inserts for waits and turn profiles (upper bound: assume every one fires)
        const double w = cons[b * 6 + 5];
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
        ins_est[b] = (float)extra;
    }
}

// ---- chunk-interleaved, block-of-four layout of everything the passes stream ------------------------------------------
// A path's D-1 steps ("edges" e = 0 .. D-2: forward step e goes from sample e to e+1, backward step e+1 from sample e+1
// to e) are cut into NT chunks of Lc edges (Lc = ceil((D-1)/NT) rounded up to a multiple of PB = 4); chunk c owns edges
// [c*Lc, min((c+1)*Lc, D-1)).  Thread c of a pass CTA walks chunk c, so at any moment the warp needs edge s of 32 different
// chunks.  The per-edge data is stored in BLOCKS of four consecutive rows of one chunk:
//      slot(e) = ((r / 4) * NT + c) * 4 + r % 4          r = e % Lc (row = position inside the chunk), c = e / Lc (column)
// so a lane's four consecutive steps are one 32-byte sector (fetched with two 16-byte loads), a warp-wide load is one
// contiguous run of memory, and -- what the earlier row-interleaved layout (slot = r * NT + c) could not give -- a lane that
// re-runs ALONE in a fix-up round fetches only sectors it uses entirely: measured with ncu on cfg2, the lone lanes of the
// fix-up rounds cost 1.2 GB per pass in that layout (8 bytes used of every 64 fetched), as much as the 96-step warm-up
// that avoids them.  Rows of RS = vap_pass_row_slots(D_cap, NT) slots per path; slot RS-1 holds the forward velocity of
// the last sample.
#define PB 4
__device__ __forceinline__ int chunk_len(int steps, int NT) { return (((steps + NT - 1) / NT) + PB - 1) & ~(PB - 1); }
__device__ __forceinline__ int edge_slot(int e, int Lc, int NT)
{
    const int c = e / Lc, r = e - c * Lc;
    return ((r >> 2) * NT + c) * PB + (r & 3);
}
// record element (row r, field f, column c) of a path: rec[((r / 4) * 4 + f) * 4 NT + 4 c + r % 4]
__device__ __forceinline__ size_t rec_index(int r, int f, int c, int NT)
{
    return ((size_t)(r >> 2) * 4 + f) * (PB * NT) + (size_t)c * PB + (r & 3);
}

// ---- pre-pass (parallel): everything of a pass step that depends neither on the velocity state nor on the events --------
// Per block of four chunk positions four field planes of 4 NT doubles: element (row s, field f, column c) of a path is
// rec[rec_index(s, f, c)]; the terms of the final sample D-1 sit in the last three doubles of the path's 4 RS.
// fields 0-2, per sample i (row / column of edge i):
//    { |kappa_i|, G_i, stat_i }
//       G_i    = min(vlim_i, cap_i)                         velocity caps (:212-218, :239)
//       stat_i = min(max_ang_acc/|k|, 2 A0/(w|k|+2), A0)    the state-independent acceleration limits for the path's own
//                (A0 when straight)                         max_acc A0 -- forward a_static AND backward d_static as long as
//                                                           no node / action point overrides max_acceleration
// field 3, per edge e:
//    gh_e = 2|theta_{e+1} - theta_e|       denominator of the wheel-acceleration term of forward step e and of backward
//                                          step e+1 (the passes make its reciprocal themselves, see recip_for_pass)
// What depends on the events is applied by the passes themselves from small shared-memory tables: the initial velocity
// v0[i+1] (regimes, stops, end velocity) enters as C_i = min(v0[i+1], G_i).  Only a path with max_acceleration overrides
// makes the pre-pass look at the regime table: stat then uses the forward regime's max_acc and the backward pass's limit
// (its max_dec) goes to a slot-order array of its own, statB.
// One thread per SLOT (coalesced stores); kappa / theta come through a shared-memory tile whose loads run along the columns.
struct SharedRecip { double b, y; bool ok; };
// a / b for several numerators over one denominator: y = RN(1/b) once, then per quotient one multiplication and two fused
// residual corrections (Markstein: with the correctly rounded reciprocal the second correction gives the correctly rounded
// quotient unless b's significand is all ones).  Operands outside the proven range take the ordinary division.
__device__ __forceinline__ SharedRecip shared_recip(double b)
{
    SharedRecip r;
    const long long bits = __double_as_longlong(b);
    r.ok = (b > 1e-150) && (b < 1e150) && ((bits & 0x000FFFFFFFFFFFFFLL) != 0x000FFFFFFFFFFFFFLL);
    r.b = b;
    r.y = 1.0 / b;
    return r;
}
__device__ __forceinline__ double div_shared(double a, const SharedRecip& r)
{
    const double aa = fabs(a);
    if (!(r.ok && aa > 1e-150 && aa < 1e150)) return a / r.b;
    double q = a * r.y;
    q = fma(fma(-r.b, q, a), r.y, q);
    q = fma(fma(-r.b, q, a), r.y, q);
    return q;
}
// does any regime of the path use a max_acc other than the path's own A0?  (max_accels[0 .. n_acc): the sampling loop's list)
__device__ __forceinline__ int pass_has_override(const double* __restrict__ ma, int n_acc, double A0)
{
    int f = 0;
    for (int j = 0; j < n_acc; j++) f |= (ma[j] != A0);
    return f;
}
__device__ __forceinline__ int last_le(const int* __restrict__ a, int n, int key)      // last j in [0, n) with a[j] <= key
{
    int lo = 0, hi = n - 1;
    while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (a[mid] <= key) lo = mid; else hi = mid - 1; }
    return lo;
}
struct SampleTerms { double ak, G, stat, stat_b; };
// acc_f: max_acc of the forward regime the sample lies in; dec_b: the backward pass's max_dec (both the path's A0 unless a
// node / action point overrides max_acceleration)
template <bool OVR>
__device__ __forceinline__ SampleTerms prepass_sample(double V, double acc_f, double dec_b, double w, double max_angular_vel,
                                                      double max_angular_accel, double k)
{
    const double ak = fabs(k);
    const bool straight = ak < 1e-6;
    // w|k| + 2 = 2 (1 + w|k|/2) bit for bit (halving and doubling are exact), so the wheel-speed cap
    // |V / (1 + w|k|/2)| (:239) IS |2V / (w|k| + 2)| (:214): one quotient serves both.
    const SharedRecip rden = shared_recip(w * ak + 2);
    const double v_kin = div_shared(2 * V, rden);
    const double cap = fabs(v_kin);
    double vlim, stat, stat_b;
    if (straight) { vlim = V; stat = acc_f; stat_b = dec_b; }
    else {
        const SharedRecip rak = shared_recip(ak);
        const double v_ang = div_shared(max_angular_vel, rak);
        const double a_ang = div_shared(max_angular_accel, rak);
        // Constraints.max_speed_at_curvature (:23-33) with 2*V/w already evaluated
        const double m = (max_angular_vel * V) / (ak * V + max_angular_vel);
        const double v_curve = pymin(m, V);
        vlim = pymin(pymin(v_ang, v_kin), v_curve);
        const double a_kin = div_shared(2 * acc_f, rden);
        stat = pymin(pymin(a_ang, a_kin), acc_f);
        stat_b = stat;
        if (OVR && dec_b != acc_f) {
            const double d_kin = div_shared(2 * dec_b, rden);
            stat_b = pymin(pymin(a_ang, d_kin), dec_b);
        }
    }
    SampleTerms t;
    t.ak = ak; t.G = pymin(vlim, cap); t.stat = stat; t.stat_b = stat_b;
    return t;
}

// ---- S3 + pre-pass: distance sampling, event candidates and the pass records in ONE kernel -------------------------------
// The sampling (distance_to_time + snap gathers, one sample per thread, lanes running along a chunk's consecutive samples)
// fills a shared-memory tile of t / theta / kappa of TC = min(NT, 64) columns x TR = 256 / TC rows, and the records are made
// from that tile one thread per slot (coalesced stores: 256 consecutive slots are whole 32-byte blocks of TC columns), so
// kappa / theta never go to HBM (t / kappa / theta are written only when the caller asks for them: inspection outputs).
// A CTA walks SP_TILES tiles DOWN the rows of its columns; a tile computes rows s0+1 .. s0+TR and takes rows s0-1 (parameter
// only: the event test needs t of the previous sample) and s0 from the tile before (the first tile computes them itself), so
// the halo costs 2 TC extra samples per CTA instead of per tile.
// The records written here use the path's own max_acc: the regimes are not known yet (k_resolve_events runs on the event
// candidates this kernel emits).  k_prepass_ovr rewrites the static limits of the paths that turn out to have overrides.
__host__ __device__ __forceinline__ int prepass_tile_cols(int NT) { return NT < 64 ? NT : 64; }
#ifndef VAP_SP_MINB
#define VAP_SP_MINB 8
#endif
#ifndef SP_TILES
#define SP_TILES 8          // 256-slot tiles per CTA of the fused sampling + pre-pass kernel
#endif
__global__ void __launch_bounds__(256, VAP_SP_MINB) k_sample_prepass(
    int N_max, int A_max, const int* __restrict__ n_nodes, const int* __restrict__ n_splines,
    const int* __restrict__ status, const double* __restrict__ cons, const double* __restrict__ ap_attr,
    const int* __restrict__ n_ap, const double* __restrict__ dgrid, int samples, long long Q_cap,
    const double* __restrict__ lut_d, const double* __restrict__ lut_t, const double* __restrict__ total_len, int spn,
    long long P_cap, const double* __restrict__ prop_k, const double* __restrict__ prop_h, long long D_cap,
    const int* __restrict__ n_samples, double* __restrict__ t_out, double* __restrict__ kap_out, double* __restrict__ th_out,
    int* __restrict__ ev_wrap, int* __restrict__ ev_nwrap, int* __restrict__ ev_apc, int* __restrict__ ev_napc,
    const int* __restrict__ lut_inv, int NT, long long RS, double* __restrict__ rec, unsigned tiles_x)
{
    extern __shared__ double s_tile[];               // two buffers of three planes (t, theta, kappa): TC columns x (TR + 2) rows
    const PathTile pt = path_tile(tiles_x);
    const long long b = pt.b;
    if (status[b] != ST_OK) return;
    const int D = n_samples[b];
    const int steps = D - 1;
    const int sh = 31 - __clz(NT);
    const int Lc = (((steps + NT - 1) >> sh) + PB - 1) & ~(PB - 1);      // chunk_len(steps, NT); NT is a power of two
    const int jend = Lc << sh;
    int j0 = pt.x * (blockDim.x * SP_TILES);
    if (steps <= 0 || j0 >= jend) return;
    const int n = n_nodes[b];
    const double* ld = lut_d + (size_t)b * Q_cap;
    const double* lt = lut_t + (size_t)b * Q_cap;
    const int Q = samples * n_splines[b];
    const double L = total_len[b];
    // per-path constants that cost divisions: made by ONE thread, published with the first tile's barrier
    __shared__ double s_c[4];
    if (threadIdx.x == 0) {
        const PropGrid g0 = prop_grid(spn, n);
        const double V_ = cons[b * 6 + 0], A0_ = cons[b * 6 + 1], w_ = cons[b * 6 + 5];
        s_c[0] = 2 * V_ / w_;                        // max_angular_vel   (:81)
        s_c[1] = 2 * A0_ / w_;                       // max_angular_accel (:82)
        s_c[2] = g0.step; s_c[3] = g0.inv_step;
    }
    __syncthreads();
    PropGrid pg;
    pg.P = spn * n; pg.n = n; pg.step = s_c[2]; pg.inv_step = s_c[3];
    const int* inv = lut_inv ? lut_inv + (size_t)b * (Q_cap + LUT_INV_HDR + 2) : nullptr;
    const double* pk = prop_k + (size_t)b * P_cap;
    const double* ph = prop_h + (size_t)b * P_cap;
    const double tn = (double)(n - 1);
    // parameter of sample x (clamped to the last sample, whose parameter is N-1 by definition, :165-176)
    auto t_of = [&](int x) {
        if (x >= D - 1) return tn;
        const double d = dgrid[x];
        return inv ? distance_to_time_inv(ld, lt, inv, Q, L, n, d) : distance_to_time32(ld, lt, Q, L, n, d);
    };
    const int tcsh = sh < 6 ? sh : 6;                // TC = min(NT, 64) columns x TR = 256 / TC rows per tile
    const int TC = 1 << tcsh;
    const int trsh = 8 - tcsh;
    const int TR = 1 << trsh;
    const int st = (TR + 2) | 1;                     // odd stride; row r of the tile sits at index r + 1 (index 0: row s0-1)
    const double V = cons[b * 6 + 0], A0 = cons[b * 6 + 1], w = cons[b * 6 + 5];
    const int A = n_ap ? n_ap[b] : 0;
    double* pr = rec + (size_t)b * RS * 4;
    const int PS = PB * NT;
    const size_t orow = (size_t)b * D_cap;
    for (int it = 0; it < SP_TILES && j0 < jend; ++it, j0 += blockDim.x) {
        double* t_t = s_tile + (it & 1) * (3 * TC * st);
        double* t_th = t_t + TC * st;
        double* t_k = t_th + TC * st;
        const double* o_t = s_tile + ((it & 1) ^ 1) * (3 * TC * st);      // the tile before
        const int c0 = (j0 >> 2) & (NT - 1);         // first column of the tile (0 unless NT > 64)
        const int s0 = (j0 >> (sh + 2)) << 2;        // first row of the tile
        {
            // rows s0+1 .. s0+TR of every column: one sample per thread, lanes along a column
            const int cc = threadIdx.x >> trsh, r = threadIdx.x & (TR - 1);
            int ee = (c0 + cc) * Lc + s0 + 1 + r;
            ee = ee > D - 1 ? D - 1 : ee;
            const double t = t_of(ee);
            double k, h;
            snap_gather2_32(pk, ph, t, pg, k, h);
            VAP_CHECK(8, cc < TC && r + 2 < st && ee >= 0 && ee <= D - 1 && D <= D_cap);
            t_t[cc * st + r + 2] = t; t_th[cc * st + r + 2] = h; t_k[cc * st + r + 2] = k;
            if (t_out) {                             // inspection outputs (a sample may be computed by two columns: same value)
                t_out[orow + ee] = t; kap_out[orow + ee] = k; th_out[orow + ee] = h;
            }
            if ((int)threadIdx.x < TC) {             // rows s0-1 and s0: from the tile before, or (first tile of the CTA) computed
                const int c = c0 + threadIdx.x;
                if (it > 0 && NT <= 64) {            // same columns as the tile before (NT > 64: a CTA's tiles change columns)
                    t_t[threadIdx.x * st + 0] = o_t[threadIdx.x * st + TR];
                    t_t[threadIdx.x * st + 1] = o_t[threadIdx.x * st + TR + 1];
                    t_th[threadIdx.x * st + 1] = o_t[TC * st + threadIdx.x * st + TR + 1];
                    t_k[threadIdx.x * st + 1] = o_t[2 * TC * st + threadIdx.x * st + TR + 1];
                } else {
                    int e0 = c * Lc + s0;
                    e0 = e0 > D - 1 ? D - 1 : e0;
                    const double t0 = t_of(e0);
                    double k0, h0;
                    snap_gather2_32(pk, ph, t0, pg, k0, h0);
                    t_t[threadIdx.x * st + 1] = t0; t_th[threadIdx.x * st + 1] = h0; t_k[threadIdx.x * st + 1] = k0;
                    t_t[threadIdx.x * st + 0] = (e0 > 0) ? t_of(e0 - 1) : 0.0;        // prev_t of sample 0 is 0 (:96)
                    if (t_out && e0 == 0) { t_out[orow] = t0; kap_out[orow] = k0; th_out[orow] = h0; }
                }
            }
        }
        __syncthreads();                             // the other buffer is free again one barrier later
        const int j = j0 + threadIdx.x;
        const int c = (j >> 2) & (NT - 1);
        const int s = ((j >> (sh + 2)) << 2) + (j & 3);
        const int e = c * Lc + s;                    // this slot's edge = the sample whose terms this thread evaluates
        if (s >= Lc || e >= steps) continue;
        const int tl = (c - c0) * st + (s - s0) + 1;
        // ---- event candidates of sample e (motion_profile_generator.py:124, :142-146); e <= D-2 here
        {
            const double t = t_t[tl], tp = t_t[tl - 1];
            if (frac1(tp) > frac1(t) && t < tn) {
                const int slot = atomicAdd(ev_nwrap + b, 1);
                if (slot < N_max) ev_wrap[(size_t)b * N_max + slot] = e;
            }
            for (int q = 0; q < A; q++) {
                const double x = ap_attr[((size_t)b * A_max + q) * APA + P_T];
                if (tp < x && t >= x) {
                    const int slot = atomicAdd(ev_napc + (size_t)b * A_max + q, 1);
                    if (slot < EV_AP_CAND) ev_apc[((size_t)b * A_max + q) * EV_AP_CAND + slot] = e;
                }
            }
        }
        // ---- the records of slot j
        const double gh = 2 * fabs(t_th[tl + 1] - t_th[tl]);
        const size_t o = (size_t)(j >> (sh + 2)) * (4 * PS) + (size_t)(j & (PS - 1));
        VAP_CHECK(9, tl >= 1 && tl + 1 < TC * st && o + 3 * PS < (size_t)(4 * RS - 3) && c - c0 >= 0 && c - c0 < TC && s - s0 >= 0 && s - s0 < TR);
        const SampleTerms tm = prepass_sample<false>(V, A0, A0, w, s_c[0], s_c[1], t_k[tl]);
        pr[o] = tm.ak; pr[o + PS] = tm.G; pr[o + 2 * PS] = tm.stat; pr[o + 3 * PS] = gh;
        if (e == steps - 1) {                        // the final sample (no edge starts there): the backward pass starts on it
            double kl, hl;
            snap_gather2_32(pk, ph, tn, pg, kl, hl);
            const SampleTerms u = prepass_sample<false>(V, A0, A0, w, s_c[0], s_c[1], kl);
            pr[4 * RS - 3] = u.ak; pr[4 * RS - 2] = u.G; pr[4 * RS - 1] = u.stat;
            if (t_out) { t_out[orow + D - 1] = tn; kap_out[orow + D - 1] = kl; th_out[orow + D - 1] = hl; }
        }
    }
}

// Paths with max_acceleration overrides (node / action point): the static acceleration limits depend on the regime, which
// k_resolve_events has only now established.  Rewrites field 2 of the records (forward limit of each sample's regime) and
// fills statB (the backward pass's limit) from field 0 (|kappa|).  One CTA per path: every path without overrides leaves at once.
__global__ void __launch_bounds__(256) k_prepass_ovr(
    const int* __restrict__ status, const double* __restrict__ cons, const int* __restrict__ n_samples, int NT, long long RS,
    double* __restrict__ rec, int E_cap, const double* __restrict__ max_accels, const int* __restrict__ bidx,
    const int* __restrict__ bval, const int* __restrict__ n_ev, double* __restrict__ statB)
{
    const long long b = blockIdx.x;
    if (status[b] != ST_OK) return;
    const double A0 = cons[b * 6 + 1];
    if (!pass_has_override(max_accels + (size_t)b * E_cap, n_ev[2 * b], A0)) return;     // uniform over the CTA
    const int D = n_samples[b];
    const int steps = D - 1;
    if (steps <= 0) return;
    const int sh = 31 - __clz(NT);
    const int Lc = chunk_len(steps, NT);
    const double V = cons[b * 6 + 0], w = cons[b * 6 + 5];
    const double mav = 2 * V / w, maa = 2 * A0 / w;
    const int PS = PB * NT;
    double* pr = rec + (size_t)b * RS * 4;
    const int nb = n_ev[2 * b + 1];
    const double dec_b = max_accels[(size_t)b * E_cap + bval[(size_t)b * E_cap + nb - 1]];       // backward max_dec
    for (int j = threadIdx.x; j < (Lc << sh); j += blockDim.x) {
        const int c = (j >> 2) & (NT - 1);
        const int s = ((j >> (sh + 2)) << 2) + (j & 3);
        const int e = c * Lc + s;
        if (e >= steps) continue;
        const size_t o = (size_t)(j >> (sh + 2)) * (4 * PS) + (size_t)(j & (PS - 1));
        const double acc_f = max_accels[(size_t)b * E_cap + bval[(size_t)b * E_cap + last_le(bidx + (size_t)b * E_cap, nb, e)]];
        const SampleTerms t = prepass_sample<true>(V, acc_f, dec_b, w, mav, maa, pr[o]);
        pr[o + 2 * PS] = t.stat;
        statB[(size_t)b * RS + j] = t.stat_b;
        if (e == steps - 1) {
            const SampleTerms u = prepass_sample<true>(V, dec_b, dec_b, w, mav, maa, pr[4 * RS - 3]);
            pr[4 * RS - 1] = u.stat;
            statB[(size_t)b * RS + RS - 1] = u.stat_b;
        }
    }
}

// ---- chunk-speculative forward / backward kernels: one CTA per path, one chunk per thread ------------------------
__device__ __forceinline__ bool same_bits(double a, double b)
{
    return __double_as_longlong(a) == __double_as_longlong(b);
}

// (w_i^2 - w_{i-1}^2) / (2|dtheta|) with IEEE results for every special case, but without sending the warp through the
// slow path of the inlined division when the numerator is 0 (cruise), or the denominator is 0 (two samples snapped
// to the same table entry) or NaN (the "straight" marker of the pre-pass).  Generic path (rare inputs only).
__device__ __noinline__ double accel_ang_div(double num, double h2)
{
    bool special = !(h2 > 0.0) || num == 0.0 || !(fabs(num) < 1e300);
    double n = special ? 1.0 : num, d = special ? 1.0 : h2;
    asm volatile("" : "+d"(n), "+d"(d));   // keep nvcc from folding the selects back into the division's operands
    double q = n / d;
    if (!special) return q;
    const double qnan = __longlong_as_double(0x7ff8000000000000LL);
    const double inf = __longlong_as_double(0x7ff0000000000000LL);
    if (h2 > 0.0) {
        if (num == 0.0) return num;                      // +-0 / positive
        return (num != num) ? qnan : copysign(inf, num); // |num| >= 1e300 or inf: overflow / inf / NaN, as IEEE '/' gives
    }
    if (h2 == 0.0) {                                     // x / +0
        if (num > 0.0) return inf;
        if (num < 0.0) return -inf;
        return qnan;                                     // 0/0 or NaN/0
    }
    return qnan;                                         // NaN denominator (the pre-pass's "straight" marker)
}

// Reciprocal of the division's denominator g = 2|dtheta|.  It does not depend on the velocity state, so the passes make it
// off the chain -- the lockstep sweeps for the four steps of a ring stage at once when the stage lands, the fix-up re-runs
// for a pair of steps two steps after loading it -- and the state-dependent chain of a step holds one multiplication and
// two fused residual corrections instead of a reciprocal refinement:
//    > 0 and finite : RN(1/g), g a normal number whose significand is not all ones (Markstein's exception)
//    +inf           : g == 0 (two samples snapped to the same heading entry; ~44 % of the samples)
//    -1             : anything else (g NaN / subnormal / all-ones significand): the pass takes the generic division
__device__ __forceinline__ double recip_for_pass(double g)
{
    const long long bits = __double_as_longlong(g);
    const bool safe = (g >= 2.2250738585072014e-308) && (g < 1e300) &&
                      ((bits & 0x000FFFFFFFFFFFFFLL) != 0x000FFFFFFFFFFFFFLL);
    double d = safe ? g : 1.0;
    asm volatile("" : "+d"(d));            // the division must never see the special values (warp-wide slow path)
    const double r = 1.0 / d;
    return safe ? r : ((g == 0.0) ? __longlong_as_double(0x7ff0000000000000LL) : -1.0);
}
__device__ __forceinline__ double2 recip_for_pass(double2 g) { return make_double2(recip_for_pass(g.x), recip_for_pass(g.y)); }

// num / h2 given rce = recip_for_pass(h2) (or NaN when h2 is the straight marker).  q0 = num * r, then two residual
// corrections: after the first the quotient is faithful, and with the correctly rounded reciprocal one more gives the
// correctly rounded quotient (Markstein), i.e. exactly what '/' returns (the sign of a zero quotient is not kept; it
// cannot reach any output).  h2 == 0 and the straight marker fall out of the multiplication: x * inf and x * NaN are
// what x / 0 and x / NaN give.  tests/test_gpu_parity.py::test_recip_division_is_ieee checks 2^30 random pairs.
__device__ __forceinline__ double accel_ang_fast(double num, double h2, double rce)
{
    const double q0 = num * rce;
    double q = fma(fma(-h2, q0, num), rce, q0);
    q = fma(fma(-h2, q, num), rce, q);
    const bool corr = rce <= 1.7976931348623157e308;          // false for NaN and +inf
    const double an = fabs(num);
    const bool in_range = (an < 1e200) && ((an > 1e-200) || (num == 0.0));
    if (rce < 0.0 || (corr && !in_range)) return accel_ang_div(num, h2);     // never taken on sane inputs
    return corr ? q : q0;
}

// One pass step from the hoisted terms.  ak = |kappa| of the step's sample, gh / rg the wheel-acceleration denominator and
// its reciprocal, stat the state-independent acceleration limit, cap the state-independent velocity limit (already merged
// with the initial / forward velocity), sq carries (v|kappa|)^2 of the previous step.
// forward step i -> i+1 (motion_profile_generator.py:193-249): |accel_ang| into the wheel term
__device__ __forceinline__ double fwd_step(double ak, double gh, double rg, double stat, double cap, double v, double& sq,
                                           double acc, double hw, double dd)
{
    const double ang_vel = v * ak;
    const double sqn = ang_vel * ang_vel;
    const double rce = (ak < 1e-6) ? __longlong_as_double(0x7ff8000000000000LL) : rg;   // straight: the term is ignored
    const double accel_ang = accel_ang_fast(sqn - sq, gh, rce);
    const double x = fabs(accel_ang) * hw;                   // ang * w / 2: halving is exact, so (ang*w)/2 == ang*(w/2)
    const double l = acc + x, rr = acc - x;                  // wheel_accel (:52-59)
    double a_wheel = (fabs(l) < fabs(rr)) ? l : rr;
    if (a_wheel < 0) a_wheel = 0;
    const double a = pymin(stat, a_wheel);
    const double s = sqrt(v * v + 2 * a * dd);
    sq = sqn;
    return pymin(cap, s);
}
// backward step i -> i-1 (:255-311): signed accel_ang; cap = min(vel_f[i-1], G_i)
__device__ __forceinline__ double bwd_step(double ak, double gh, double rg, double stat, double cap, double v, double& sq,
                                           double acc, double hw, double dd)
{
    const double ang_vel = v * ak;
    const double sqn = ang_vel * ang_vel;
    const double rce = (ak < 1e-6) ? __longlong_as_double(0x7ff8000000000000LL) : rg;
    const double accel_ang = accel_ang_fast(sqn - sq, gh, rce);
    const double x = accel_ang * hw;
    const double l = acc + x, rr = acc - x;
    double a_wheel = (fabs(l) < fabs(rr)) ? l : rr;
    if (a_wheel < 0) a_wheel = 0;
    const double dcl = pymin(stat, a_wheel);
    const double pv = sqrt(v * v + 2 * dcl * dd);
    sq = sqn;
    return pymin(pv, cap);
}

// ------------------------------------------------------------------------------------------------------------------
// Chunk-speculative passes: CTA = one path, thread c = chunk c (blockDim.x chunks).
//
// Sweep 1: every thread runs its own chunk from a guessed state (lockstep, all lanes busy).  Fix-up rounds: a chunk whose
// predecessor's end state differs bitwise from the state it started from re-runs from the true state; the re-run stops as
// soon as two consecutive velocities equal the stored ones bitwise (from there the old values ARE the serial values).
// Rounds end when no chunk had to re-run; then, by induction from chunk 0, every value is the serial value.
//
// The kernels are bound by the latency of the dependent fp64 chain of one step, so they are written for a short chain:
// event tables in shared memory, 32-bit indices, the division's reciprocal made off the chain, coalesced slot-order streams.
// The lockstep first sweep takes its records from a per-warp shared-memory ring that TMA bulk copies fill a whole block
// ahead; the fix-up re-runs and the warm-up are out of line and load their records one pair ahead themselves.
// ------------------------------------------------------------------------------------------------------------------
#define CH_INT_MAX 2147483647
#ifndef VAP_PASS_REGS_TMA
#define VAP_PASS_REGS_TMA 112 // 112 x 32 registers allow 18 one-warp CTAs per SM; with cfg2's tables the shared-memory rings (8 KB
                              // forward, 10 KB backward per warp) allow 21 / 18.  Fewer registers make the out-of-line re-run
                              // functions spill more (96: 3.69 ms per cfg2 step, 112: 3.47, 128: 3.56)
#endif

// 16-byte read-only load of two consecutive doubles
__device__ __forceinline__ double2 ldg_d2(const double* p) { return __ldg(reinterpret_cast<const double2*>(p)); }
__device__ __forceinline__ void st_d2(double* p, double x, double y) { *reinterpret_cast<double2*>(p) = make_double2(x, y); }

// a lone lane of a fix-up re-run asks the L2 for the sectors it will need a few blocks on (its own loads only look two steps
// ahead, which does not cover an HBM round trip; the lockstep sweeps have the TMA ring for that)
#define RERUN_PF 4
__device__ __forceinline__ void l2_prefetch(const void* g) { asm volatile("prefetch.global.L2 [%0];" ::"l"(g)); }

// contribution of one step to the travel-time estimate (single precision: it only sizes buffers)
__device__ __forceinline__ float t_est_term(double va, double vb, float dd_over_dt)
{
    const float vm = 0.5f * ((float)va + (float)vb);
    return __fdividef(dd_over_dt, fmaxf(vm, 0.05f));
}

// per-path event tables of the forward pass in shared memory
struct FwdTables {
    const int* bi; const double* acc; int n_b;       // max_acc regimes: acc[j] from sample bi[j] on
    const int* vi; const double* vv; int n_v;        // initial velocity: vv[j] from sample vi[j] on (stops / end included)
};

// forward chunk: edges lo .. lo+len-1, lo at the first row of a block.  p points at (field 0, own column) of that block of the
// record rows, q at the same block of the forward velocities (q[r] = velocity at sample lo + r).  A lane only ever writes
// its OWN column: the velocity of sample lo+len is the start state of the next column's lane, which stores it itself; only
// the path's last chunk writes it (to the tail slot).  Records come as 16-byte pairs, two steps per pair, the next pair
// fetched while the current one is being used (two named buffers, no register rotation).  NT is a compile-time constant:
// every access is pointer + immediate.  old_end: what this lane's previous run produced for sample lo+len (RUN_RERUN).
#define RUN_RERUN 1     // fix-up: bitwise merge detection against the stored velocities
#define RUN_DRY 2       // warm-up before a speculative chunk: state only, no stores
template <int NT, int MODE>
__device__ __forceinline__ bool fwd_run(const double* __restrict__ p, double* __restrict__ q, double* __restrict__ tail,
                                        double old_end, int lo, int len, const FwdTables& T, double hw,
                                        double dd, double& v, double& sq, bool prev_same)
{
    constexpr int PS = PB * NT, BS = 4 * PS;
    constexpr bool RERUN = (MODE == RUN_RERUN);
    constexpr bool DRY = (MODE == RUN_DRY);
    int j = 0;
    while (j + 1 < T.n_b && T.bi[j + 1] <= lo) j++;
    double acc = T.acc[j];
    int nb_next = (j + 1 < T.n_b) ? T.bi[j + 1] : CH_INT_MAX;
    int jv = 0;                                      // initial velocity of sample e+1
    while (jv + 1 < T.n_v && T.vi[jv + 1] <= lo + 1) jv++;
    double v0n = T.vv[jv];
    int nv_next = (jv + 1 < T.n_v) ? T.vi[jv + 1] : CH_INT_MAX;
    int e = lo;
    const int hi = lo + len;
#define FWD_ONE(AK_, G_, ST_, GH_, RG_, OLD_)                                                                        \
        if (e == nb_next) { j++; acc = T.acc[j]; nb_next = (j + 1 < T.n_b) ? T.bi[j + 1] : CH_INT_MAX; }              \
        if (e + 1 == nv_next) { jv++; v0n = T.vv[jv]; nv_next = (jv + 1 < T.n_v) ? T.vi[jv + 1] : CH_INT_MAX; }      \
        v = fwd_step(AK_, GH_, RG_, ST_, pymin(v0n, G_), v, sq, acc, hw, dd);                                        \
        if (RERUN) {                                                                                                 \
            const bool same = same_bits(OLD_, v);                                                                    \
            if (same && prev_same) return true;       /* state equals the old run's: the rest is unchanged */        \
            prev_same = same;                                                                                        \
        }                                                                                                            \
        ++e;
    // a pair's reciprocals are made two steps after its loads, just before its own steps
    double2 akA = ldg_d2(p), GA = ldg_d2(p + PS), stA = ldg_d2(p + 2 * PS), ghA = ldg_d2(p + 3 * PS), rgA;
    double2 akB, GB, stB, ghB, rgB;
    double2 oA = make_double2(0.0, 0.0), oB = oA;    // old velocities (RERUN): pair A = samples e, e+1; pair B = e+2, e+3
    if (RERUN) oA = *reinterpret_cast<const double2*>(q);
    // whole blocks (look-ahead loads never leave the path's rows: they are padded by one block)
    if (RERUN) {
#pragma unroll
        for (int k = 1; k < RERUN_PF; k++)
            if (k < (len >> 2)) {
#pragma unroll
                for (int f = 0; f < 4; f++) l2_prefetch(p + (size_t)k * BS + f * PS);
                l2_prefetch(q + (size_t)k * PS);
            }
    }
    for (int blk = len >> 2; blk > 0; --blk) {
        if (RERUN && blk > RERUN_PF) {
#pragma unroll
            for (int f = 0; f < 4; f++) l2_prefetch(p + (size_t)RERUN_PF * BS + f * PS);
            l2_prefetch(q + (size_t)RERUN_PF * PS);
        }
        akB = ldg_d2(p + 2); GB = ldg_d2(p + PS + 2); stB = ldg_d2(p + 2 * PS + 2); ghB = ldg_d2(p + 3 * PS + 2);
        if (RERUN) oB = *reinterpret_cast<const double2*>(q + 2);
        rgA = recip_for_pass(ghA);
        const double vin = v;
        FWD_ONE(akA.x, GA.x, stA.x, ghA.x, rgA.x, oA.y)
        const double v1 = v;
        if (RERUN) st_d2(q, vin, v1);                 // a re-run may leave at any step: store as soon as a pair is complete
        FWD_ONE(akA.y, GA.y, stA.y, ghA.y, rgA.y, oB.x)
        const double v2 = v;
        p += BS;
        akA = ldg_d2(p); GA = ldg_d2(p + PS); stA = ldg_d2(p + 2 * PS); ghA = ldg_d2(p + 3 * PS);
        if (RERUN) oA = *reinterpret_cast<const double2*>(q + PS);
        rgB = recip_for_pass(ghB);
        FWD_ONE(akB.x, GB.x, stB.x, ghB.x, rgB.x, oB.y)
        if (RERUN) st_d2(q + 2, v2, v);
        FWD_ONE(akB.y, GB.y, stB.y, ghB.y, rgB.y, ((e + 1 < hi) ? oA.x : old_end))
        q += PS;
    }
    // ragged end of the path's last chunk: up to three more edges, one at a time (their rows are in the A pairs / row 2)
    if (e < hi) {
        if (!DRY) q[0] = v;
        const int rem = hi - e;
        rgA = recip_for_pass(ghA);
        {
            const double old = RERUN ? ((rem > 1) ? oA.y : old_end) : 0.0;
            FWD_ONE(akA.x, GA.x, stA.x, ghA.x, rgA.x, old)
            if (!DRY && e < hi) q[1] = v;
        }
        if (e < hi) {
            const double old = RERUN ? ((rem > 2) ? q[2] : old_end) : 0.0;
            FWD_ONE(akA.y, GA.y, stA.y, ghA.y, rgA.y, old)
            if (!DRY && e < hi) q[2] = v;
        }
        if (e < hi) {
            const double a2 = __ldg(p + 2), g2 = __ldg(p + PS + 2), s2 = __ldg(p + 2 * PS + 2), h2 = __ldg(p + 3 * PS + 2);
            FWD_ONE(a2, g2, s2, h2, recip_for_pass(h2), old_end)
        }
    }
#undef FWD_ONE
    if (!DRY && tail) *tail = v;
    return false;
}

// ---- sweeps staged through shared memory by TMA -------------------------------------------------------------------------
// In the block-of-four layout the share of one WARP (32 columns) in one block row is a contiguous 1 KB per field plane, so
// the lockstep first sweep does not load records into registers at all: one lane issues one cp.async.bulk per plane and
// block row (four for the forward pass; five for the backward pass, which also streams the forward velocities) into a
// two-stage shared-memory ring that completes on an mbarrier, a whole block (four steps) ahead of its use.  When a stage has
// landed, each lane makes the reciprocals of its four gh values together (kept in registers) and then takes everything
// else of a step from shared memory.  Nothing of the stream passes through L1, no look-ahead buffers live in registers, and
// the HBM reads are 1 KB bursts issued thousands of cycles before they are needed.
#define TMA_PLANE_DOUBLES (PB * 32)                    // one plane of one stage: 32 columns x 4 rows
struct WarpRing {
    double* stage;       // this warp's two stages
    unsigned bar;        // shared-memory address of its two mbarriers
    int planes;          // field planes per stage (4 forward, 5 backward)
    unsigned bytes;      // bytes of one plane copy (32 bytes per column of the warp)
#ifdef VAP_BOUNDS_CHECK
    const double *rec_lo, *rec_hi, *x_lo, *x_hi;     // the path's record rows / slot-order rows (forward velocities, override limits)
    unsigned smem_lo, smem_hi, bar_hi;               // the CTA's rings; its mbarriers sit behind them
#endif
};
// lane 0: refill stage `s` with block row `rb`; src[f] = plane f of block row 0 at the warp's first column, strides in doubles
template <int NT>
__device__ __forceinline__ void ring_issue(const WarpRing& R, int s, const double* rec_row0, const double* x_row0,
                                           const double* sb_row0, int rb)
{
    constexpr int PS = PB * NT, BS = 4 * PS;
    const unsigned bar = R.bar + 8 * s;
    const unsigned dst = (unsigned)__cvta_generic_to_shared(R.stage + (size_t)s * R.planes * TMA_PLANE_DOUBLES);
    fence_proxy_async();                                   // the lanes' reads of this stage precede the TMA writes
    mbar_expect_tx(bar, R.bytes * R.planes);
    const double* src = rec_row0 + (size_t)rb * BS;
    if (NT == 32 && !sb_row0) {
        // 32 chunks: the four planes of a block row are contiguous in memory and in the stage: ONE 4 KB copy
#ifdef VAP_BOUNDS_CHECK
        VAP_CHECK(1, rb >= 0 && src >= R.rec_lo && src + 4 * R.bytes / 8 <= R.rec_hi && (reinterpret_cast<uintptr_t>(src) & 15) == 0);
        VAP_CHECK(2, dst >= R.smem_lo && dst + 4 * R.bytes <= R.smem_hi && bar >= R.smem_hi && bar + 8 <= R.bar_hi);
#endif
        bulk_g2s(dst, src, 4 * R.bytes, bar);
    } else
#pragma unroll
    for (int f = 0; f < 4; f++) {
        const double* g = (f == 2 && sb_row0) ? sb_row0 + (size_t)rb * PS : src + f * PS;
#ifdef VAP_BOUNDS_CHECK
        if (f == 2 && sb_row0) VAP_CHECK(0, rb >= 0 && (reinterpret_cast<uintptr_t>(g) & 15) == 0);
        else VAP_CHECK(1, rb >= 0 && g >= R.rec_lo && g + R.bytes / 8 <= R.rec_hi && (reinterpret_cast<uintptr_t>(g) & 15) == 0);
        VAP_CHECK(2, dst + f * TMA_PLANE_DOUBLES * 8 >= R.smem_lo && dst + f * TMA_PLANE_DOUBLES * 8 + R.bytes <= R.smem_hi && bar >= R.smem_hi && bar + 8 <= R.bar_hi);
#endif
        bulk_g2s(dst + f * TMA_PLANE_DOUBLES * 8, g, R.bytes, bar);
    }
    if (x_row0) {
#ifdef VAP_BOUNDS_CHECK
        VAP_CHECK(3, x_row0 + (size_t)rb * PS >= R.x_lo && x_row0 + (size_t)rb * PS + R.bytes / 8 <= R.x_hi);
        VAP_CHECK(2, dst + 4 * TMA_PLANE_DOUBLES * 8 + R.bytes <= R.smem_hi);
#endif
        bulk_g2s(dst + 4 * TMA_PLANE_DOUBLES * 8, x_row0 + (size_t)rb * PS, R.bytes, bar);
    }
}

// forward first sweep of one warp: every lane walks its chunk (edges lo .. lo+len-1; len = 0 for an idle lane) in lockstep.
// rec_w: field 0 of block row 0 at the warp's first column; lc: this lane's column minus the warp's first; q: own column of
// the forward velocities (block row 0).
template <int NT>
__device__ __forceinline__ void fwd_sweep_tma(const WarpRing& R, const double* __restrict__ rec_w, int lc, double* __restrict__ q,
                                              double* __restrict__ tail, int lo, int len, const FwdTables& T, double hw,
                                              double dd, double& v, double& sq)
{
    constexpr int PS = PB * NT;
    constexpr int PD = TMA_PLANE_DOUBLES;
    const int lane = threadIdx.x & 31;
    const int nbw = __reduce_max_sync(0xffffffffu, (len + PB - 1) >> 2);      // block rows the warp streams
    if (lane == 0) {
        if (nbw > 0) ring_issue<NT>(R, 0, rec_w, nullptr, nullptr, 0);
        if (nbw > 1) ring_issue<NT>(R, 1, rec_w, nullptr, nullptr, 1);
    }
    int j = 0;
    while (j + 1 < T.n_b && T.bi[j + 1] <= lo) j++;
    double acc = T.acc[j];
    int nb_next = (j + 1 < T.n_b) ? T.bi[j + 1] : CH_INT_MAX;
    int jv = 0;                                      // initial velocity of sample e+1
    while (jv + 1 < T.n_v && T.vi[jv + 1] <= lo + 1) jv++;
    double v0n = T.vv[jv];
    int nv_next = (jv + 1 < T.n_v) ? T.vi[jv + 1] : CH_INT_MAX;
    int e = lo;
    const int hi = lo + len;
    const int nfull = len >> 2;
#define FWD_T(ROW_)                                                                                                  \
        {                                                                                                            \
            const double ak_ = S[ROW_], G_ = S[PD + ROW_], st_ = S[2 * PD + ROW_], gh_ = gh[ROW_], rg_ = rg[ROW_];    \
            if (e == nb_next) { j++; acc = T.acc[j]; nb_next = (j + 1 < T.n_b) ? T.bi[j + 1] : CH_INT_MAX; }          \
            if (e + 1 == nv_next) { jv++; v0n = T.vv[jv]; nv_next = (jv + 1 < T.n_v) ? T.vi[jv + 1] : CH_INT_MAX; }  \
            v = fwd_step(ak_, gh_, rg_, st_, pymin(v0n, G_), v, sq, acc, hw, dd);                                    \
            ++e;                                                                                                     \
        }
    for (int blk = 0; blk < nbw; ++blk) {
        const int s = blk & 1;
        mbar_wait(R.bar + 8 * s, (blk >> 1) & 1);
        const double* S = R.stage + (size_t)s * 4 * PD + lc * PB;
        VAP_CHECK(6, lc >= 0 && lc < 32 && (unsigned)__cvta_generic_to_shared(S + 3 * PD + 3) + 8 <= R.smem_hi);
        double gh[PB], rg[PB];
#pragma unroll
        for (int r = 0; r < PB; r++) gh[r] = S[3 * PD + r];
#pragma unroll
        for (int r = 0; r < PB; r++) rg[r] = recip_for_pass(gh[r]);
        if (blk < nfull) {                           // a whole block of this lane's chunk
            const double vin = v;
            FWD_T(0)
            const double v1 = v;
            FWD_T(1)
            const double v2 = v;
            FWD_T(2)
            st_d2(q, vin, v1); st_d2(q + 2, v2, v);  // samples e0 .. e0+3: the whole 32-byte sector
            FWD_T(3)
            q += PS;
        } else if (e < hi) {                         // ragged end of the path's last chunk: up to three edges
            q[0] = v;
            FWD_T(0)
            if (e < hi) { q[1] = v; FWD_T(1) }
            if (e < hi) { q[2] = v; FWD_T(2) }
        }
        __syncwarp();
        if (lane == 0 && blk + 2 < nbw) ring_issue<NT>(R, s, rec_w, nullptr, nullptr, blk + 2);
    }
#undef FWD_T
    if (tail && len > 0) *tail = v;
}

// The fix-up re-runs and the warm-up run are cold, divergent code: out of line, so that their registers do not count against
// the lockstep sweep (state goes through a two-element array).
template <int NT>
__device__ __noinline__ bool fwd_rerun(const double* p, double* q, double* tail, double old_end, int lo, int len, FwdTables T,
                                       double hw, double dd, double* st, bool prev_same)
{
    double v = st[0], sq = st[1];
    const bool merged = fwd_run<NT, RUN_RERUN>(p, q, tail, old_end, lo, len, T, hw, dd, v, sq, prev_same);
    st[0] = v; st[1] = sq;
    return merged;
}
template <int NT>
__device__ __noinline__ void fwd_dry(const double* p, int lo, int len, FwdTables T, double hw, double dd, double* st)
{
    double v = st[0], sq = st[1];
    fwd_run<NT, RUN_DRY>(p, nullptr, nullptr, 0.0, lo, len, T, hw, dd, v, sq, false);
    st[0] = v; st[1] = sq;
}

// Forward pass.  Chunk c = thread c.  vfT: forward velocities in slot order (vfT[slot(e)] = velocity at sample e), the
// velocity of the last sample in slot RS-1.
template <int NT>
__global__ void __maxnreg__(VAP_PASS_REGS_TMA) k_fwd_chunked(
    const int* __restrict__ status, const double* __restrict__ cons, double dd, double start_vel, double end_vel,
    long long RS, const int* __restrict__ n_samples, const double* __restrict__ rec, int E_cap,
    const double* __restrict__ max_accels, const int* __restrict__ bidx, const int* __restrict__ bval,
    const int* __restrict__ n_ev, const int* __restrict__ vr_idx, const double* __restrict__ vr_val,
    const int* __restrict__ st_idx, const int* __restrict__ n_vr, double* __restrict__ vfT, int* __restrict__ rounds_out,
    int warm, int max_rounds, int ring_off)
{
    extern __shared__ __align__(128) unsigned char s_mem[];
    const int c = threadIdx.x;
    const long long b = blockIdx.x;
    const int VC = 3 * E_cap + 2;                                  // capacity of the initial-velocity table
    double* s_endv = reinterpret_cast<double*>(s_mem);            // [NT] end state of every chunk: v and (v|k|)^2
    double* s_endw = s_endv + NT;
    double* s_usev = s_endw + NT;                                 // [NT] start state every chunk last used
    double* s_usew = s_usev + NT;
    double* s_acc = s_usew + NT;                                  // [E_cap] max_acc of regime j
    double* s_vv = s_acc + E_cap;                                 // [VC]
    int* s_bi = reinterpret_cast<int*>(s_vv + VC);                // [E_cap] first sample of regime j
    int* s_vi = s_bi + E_cap;                                     // [VC]
    __shared__ int s_nv;
    if (status[b] != ST_OK) return;                               // uniform over the CTA
    const int D = n_samples[b];
    const int steps = D - 1;
    double* vf = vfT + (size_t)b * RS;
    if (c == 0) { vf[0] = start_vel; vf[RS - 1] = start_vel; if (rounds_out) rounds_out[2 * b] = 0; }
    if (steps <= 0) return;
    const int n_b = n_ev[2 * b + 1];
    for (int k = c; k < n_b; k += NT) {
        s_bi[k] = bidx[(size_t)b * E_cap + k];
        s_acc[k] = max_accels[(size_t)b * E_cap + bval[(size_t)b * E_cap + k]];
    }
    if (c == 0) {
        // initial velocity v0[x] as one sorted breakpoint table (motion_profile_generator.py:95-176): the regime value from
        // vr_idx[j] on, 0.01 at the stop samples, end_vel at the last sample.  Three sorted streams (regime starts, stops,
        // sample after a stop) are merged; the value at a breakpoint follows the reference's order of overwrites.
        const int* vi = vr_idx + (size_t)b * E_cap;
        const double* vv = vr_val + (size_t)b * E_cap;
        const int* si = st_idx + (size_t)b * E_cap;
        const int nvr = n_vr[2 * b], nst = n_vr[2 * b + 1];
        int pv = 0, ps = 0, pa = 0, n = 0, reg = 0;
        while (true) {
            int x = CH_INT_MAX;
            if (pv < nvr) x = vi[pv];
            if (ps < nst && si[ps] < x) x = si[ps];
            if (pa < nst && si[pa] + 1 < x) x = si[pa] + 1;
            if (x >= D - 1) break;
            bool stop = false;
            while (pv < nvr && vi[pv] == x) { reg = pv; pv++; }
            while (ps < nst && si[ps] == x) { stop = true; ps++; }
            while (pa < nst && si[pa] + 1 == x) pa++;
            s_vi[n] = x; s_vv[n] = stop ? 0.01 : vv[reg]; n++;
        }
        s_vi[n] = D - 1; s_vv[n] = end_vel; n++;
        s_nv = n;
    }
    const int Lc = chunk_len(steps, NT);
    const int nch = (steps + Lc - 1) / Lc;
    const bool active = c < nch;
    const int lo = c * Lc;
    const int len = (lo + Lc < steps) ? Lc : steps - lo;
    const double* P = rec + (size_t)b * RS * 4;
    double* tail = (active && lo + len == steps) ? vf + (RS - 1) : nullptr;  // only the last chunk stores the final sample
    const double hw = cons[b * 6 + 5] * 0.5;
    // every warp owns a two-stage ring (4 planes of 1 KB per stage) and two mbarriers behind the tables
    WarpRing R;
    constexpr int WARPS = (NT + 31) / 32;
    const int w = c >> 5;
    R.stage = reinterpret_cast<double*>(s_mem + ring_off) + (size_t)w * 2 * 4 * TMA_PLANE_DOUBLES;
    R.bar = (unsigned)__cvta_generic_to_shared(s_mem + ring_off + (size_t)WARPS * 2 * 4 * TMA_PLANE_DOUBLES * 8 + 16 * w);
    R.planes = 4;
    R.bytes = (NT < 32 ? NT : 32) * PB * 8;
#ifdef VAP_BOUNDS_CHECK
    R.rec_lo = P; R.rec_hi = P + 4 * RS; R.x_lo = R.x_hi = nullptr;
    R.smem_lo = (unsigned)__cvta_generic_to_shared(s_mem + ring_off);
    R.smem_hi = R.smem_lo + WARPS * 2 * 4 * TMA_PLANE_DOUBLES * 8;
    R.bar_hi = R.smem_hi + 16 * WARPS;
#endif
    if ((c & 31) == 0) { mbar_init(R.bar, 1); mbar_init(R.bar + 8, 1); fence_mbar_init(); }
    __syncthreads();
    FwdTables T;
    T.bi = s_bi; T.acc = s_acc; T.n_b = n_b; T.vi = s_vi; T.vv = s_vv; T.n_v = s_nv;

    // ---- sweep 1: chunk c > 0 may start `wl` steps BEFORE its own range (in the previous column) from the guess "the state-
    // independent caps bind on the two samples before that point": v[s0] = C[s0-1] = min(v0[s0], G[s0-1]) and
    // omega_prev = C[s0-2] |kappa[s0-1]|, and only compute (no stores) until it reaches its range.  In this layout a fix-up
    // re-run costs only the sectors it uses, which is less than the warm-up reads: the default is no warm-up.
    // (Exactness never depends on the guess: the rounds below verify bitwise.)
    {
        double v = start_vel, sq = 0.0;
        if (active) {
            if (c > 0) {
                auto v0_at = [&](int x) { int q = 0; while (q + 1 < T.n_v && T.vi[q + 1] <= x) q++; return T.vv[q]; };
                auto term = [&](int x, int fld) { const int cx = x / Lc, rx = x - cx * Lc; return __ldg(P + rec_index(rx, fld, cx, NT)); };
                int wl = warm < Lc ? warm : Lc;                      // the warm-up stays inside the previous column
                if (wl > lo - 2) wl = lo - 2 > 0 ? lo - 2 : 0;
                wl &= ~(PB - 1);                                     // ... and starts on a block
                const int s0 = lo - wl;
                const double vm1 = (s0 >= 2) ? pymin(v0_at(s0 - 1), term(s0 - 2, 1)) : start_vel;
                v = pymin(v0_at(s0), term(s0 - 1, 1));
                const double wp = vm1 * term(s0 - 1, 0);
                sq = wp * wp;
                if (wl > 0) {
                    double st[2] = {v, sq};
                    fwd_dry<NT>(P + rec_index(Lc - wl, 0, c - 1, NT), s0, wl, T, hw, dd, st);
                    v = st[0]; sq = st[1];
                }
            }
            s_usev[c] = v; s_usew[c] = sq;
            // extent of what this lane's runs touch (look-ahead block included): record rows and forward-velocity row
            VAP_CHECK(4, c * PB + PB <= PB * NT && (size_t)(((len + 3) >> 2) + 1) * 4 * PB * NT <= (size_t)(4 * RS - 3) &&
                             (size_t)(((len + 3) >> 2) + 1) * PB * NT <= (size_t)(RS - 1) && lo + len <= steps);
        }
        fwd_sweep_tma<NT>(R, P + (c & ~31) * PB, c & 31, vf + c * PB, tail, lo, active ? len : 0, T, hw, dd, v, sq);
        s_endv[c] = v; s_endw[c] = sq;
    }
    __syncthreads();

    // ---- fix-up rounds
    int rounds = 0;
    for (int round = 1; round < NT && round <= max_rounds; round++) {
        bool need = false;
        double in_v = 0.0, in_w = 0.0;
        if (active && c >= round) {
            in_v = s_endv[c - 1]; in_w = s_endw[c - 1];
            need = !(same_bits(in_v, s_usev[c]) && same_bits(in_w, s_usew[c]));
        }
        if (!__syncthreads_or(need)) break;          // also orders this round's reads before its writes
        rounds = round;
        if (need) {
            double st[2] = {in_v, in_w};
            const bool merged = fwd_rerun<NT>(P + c * PB, vf + c * PB, tail, s_endv[c], lo, len, T, hw, dd, st,
                                              same_bits(in_v, s_usev[c]));
            s_usev[c] = in_v; s_usew[c] = in_w;
            if (!merged) { s_endv[c] = st[0]; s_endw[c] = st[1]; }
        }
        __syncthreads();
    }
    if (c == 0 && rounds_out) rounds_out[2 * b] = rounds;
}

// backward chunk: edges lo+len-1 down to lo (lo at the first row of a block).  p / f / sb point at (field 0, own column) of the
// chunk's FIRST block of the record rows / forward velocities / override limits, o at sample lo of the path's final
// velocities, which this pass writes in SAMPLE order (16-byte pairs: the time stage and the API read them as they are).
// Edge e = lo + r (the reference's step i = e+1 -> e) uses the terms of sample e+1 (fields 0-2 of row r+1: carried over from
// the pair above; for the chunk's top edge the three `top` values), gh (field 3) of row r with its reciprocal, and the
// forward velocity of row r, and writes the final velocity of sample e.
// OVR: the path has max_acceleration overrides; the static limit of the backward pass then comes from its own slot-order
// array `sb` (same slots as the forward velocities) instead of field 2 of the record rows.
template <int NT, int MODE, bool OVR>
__device__ __forceinline__ bool bwd_run(const double* __restrict__ p, const double* __restrict__ f, double* __restrict__ o,
                                        const double* __restrict__ sb, int lo, int len, double top_ak, double top_G,
                                        double top_st, const int* s_bi, const double* s_acc, int n_b, double acc0, double hw,
                                        double dd, double& v, double& sq, bool prev_same, float& est, float dd_over_dt,
                                        double old_top = 0.0)
{
    constexpr int PS = PB * NT, BS = 4 * PS;
    constexpr bool RERUN = (MODE == RUN_RERUN);
    constexpr bool DRY = (MODE == RUN_DRY);
    // regime at the chunk start (walking down from D-1): the smallest boundary index > i was the last one applied
    int e = lo + len - 1;                            // current edge; the reference's loop index is i = e + 1
    int j = n_b - 1;
    double acc = acc0;
    while (j >= 0 && s_bi[j] > e + 1) { acc = s_acc[j]; j--; }
    int nb_next = (j >= 0) ? s_bi[j] : -1;
    // est: travel-time estimate of the chunk's edges, kept up to date by the re-runs (new term minus old term per step; OLDUP_
    // is the stored velocity of the sample above the step's)
#define BWD_ONE(AK_, G_, ST_, GH_, RG_, F_, OLD_, OLDUP_)                                                            \
        if (e + 1 == nb_next) { acc = s_acc[j]; j--; nb_next = (j >= 0) ? s_bi[j] : -1; }                             \
        {                                                                                                            \
            const double vup = v;                                                                                    \
            v = bwd_step(AK_, GH_, RG_, ST_, pymin(F_, G_), v, sq, acc, hw, dd);                                     \
            if (!DRY) est += t_est_term(vup, v, dd_over_dt);                                                         \
            if (RERUN) est -= t_est_term(OLDUP_, OLD_, dd_over_dt);                                                  \
        }                                                                                                            \
        if (RERUN) {                                                                                                 \
            const bool same = same_bits(OLD_, v);                                                                    \
            if (same && prev_same) return true;                                                                      \
            prev_same = same;                                                                                        \
        }                                                                                                            \
        --e;
    int blk = len >> 2;                              // whole blocks below the ragged top
    p += (size_t)blk * BS; f += (size_t)blk * PS; sb += (size_t)blk * PS; if (!DRY) o += blk * PB;
    double tak = top_ak, tG = top_G, tst = top_st;   // terms of sample e+1
    double oup = old_top;                            // velocity of sample e+1 in this lane's previous run (its start state then)
    // ragged top of the path's last chunk: up to three edges (rows 4 blk + rem-1 .. 4 blk), one at a time
    for (int r = (len & 3) - 1; r >= 0; --r) {
        const double gh = __ldg(p + 3 * PS + r), fv = __ldg(f + r);
        const double old = RERUN ? o[r] : 0.0;
        BWD_ONE(tak, tG, tst, gh, recip_for_pass(gh), fv, old, oup)
        if (!DRY) o[r] = v;
        oup = old;
        tak = __ldg(p + r); tG = __ldg(p + PS + r); tst = OVR ? __ldg(sb + r) : __ldg(p + 2 * PS + r);
    }
    if (blk == 0) return false;
    // whole blocks, top down: pair B (rows 2, 3) then pair A (rows 0, 1) of each; the next pair is fetched while the current
    // one is being used, and its reciprocals are made two steps later, just before its own steps
    p -= BS; f -= PS; sb -= PS; if (!DRY) o -= PB;
    if (RERUN) {
#pragma unroll
        for (int k = 1; k < RERUN_PF; k++)
            if (k < blk) {
#pragma unroll
                for (int fl = 0; fl < 4; fl++) if (!(OVR && fl == 2)) l2_prefetch(p - (size_t)k * BS + fl * PS);
                l2_prefetch(f - (size_t)k * PS);
                l2_prefetch(o - k * PB);
                if (OVR) l2_prefetch(sb - (size_t)k * PS);
            }
    }
    double2 akB = ldg_d2(p + 2), GB = ldg_d2(p + PS + 2), stB = OVR ? ldg_d2(sb + 2) : ldg_d2(p + 2 * PS + 2),
            ghB = ldg_d2(p + 3 * PS + 2), fB = ldg_d2(f + 2);
    double2 akA, GA, stA, ghA, fA;
    double2 oA = make_double2(0.0, 0.0), oB = oA;
    if (RERUN) oB = *reinterpret_cast<const double2*>(o + 2);
    while (true) {
        if (RERUN && blk > RERUN_PF) {
#pragma unroll
            for (int fl = 0; fl < 4; fl++) if (!(OVR && fl == 2)) l2_prefetch(p - (size_t)RERUN_PF * BS + fl * PS);
            l2_prefetch(f - (size_t)RERUN_PF * PS);
            l2_prefetch(o - RERUN_PF * PB);
            if (OVR) l2_prefetch(sb - (size_t)RERUN_PF * PS);
        }
        akA = ldg_d2(p); GA = ldg_d2(p + PS); stA = OVR ? ldg_d2(sb) : ldg_d2(p + 2 * PS); ghA = ldg_d2(p + 3 * PS);
        fA = ldg_d2(f);
        if (RERUN) oA = *reinterpret_cast<const double2*>(o);
        const double2 rgB = recip_for_pass(ghB);
        BWD_ONE(tak, tG, tst, ghB.y, rgB.y, fB.y, oB.y, oup)
        const double v3 = v;
        BWD_ONE(akB.y, GB.y, stB.y, ghB.x, rgB.x, fB.x, oB.x, oB.y)
        const double v2 = v;
        if (RERUN) st_d2(o + 2, v2, v3);              // a re-run may leave at any step: store as soon as a pair is complete
        const double a2 = akB.x, g2 = GB.x, s2 = stB.x;              // terms of row 2, for the edge of row 1
        const double ob0 = oB.x;
        const bool more = --blk > 0;
        if (more) {                                                  // pair B of the block below
            akB = ldg_d2(p - BS + 2); GB = ldg_d2(p - BS + PS + 2); stB = OVR ? ldg_d2(sb - PS + 2) : ldg_d2(p - BS + 2 * PS + 2);
            ghB = ldg_d2(p - BS + 3 * PS + 2); fB = ldg_d2(f - PS + 2);
            if (RERUN) oB = *reinterpret_cast<const double2*>(o - PB + 2);
        }
        const double2 rgA = recip_for_pass(ghA);
        BWD_ONE(a2, g2, s2, ghA.y, rgA.y, fA.y, oA.y, ob0)
        const double v1 = v;
        BWD_ONE(akA.y, GA.y, stA.y, ghA.x, rgA.x, fA.x, oA.x, oA.y)
        if (RERUN) st_d2(o, v, v1);
        if (!more) break;
        oup = oA.x;
        tak = akA.x; tG = GA.x; tst = stA.x;
        p -= BS; f -= PS; sb -= PS; if (!DRY) o -= PB;
    }
#undef BWD_ONE
    return false;
}

// backward first sweep of one warp (see fwd_sweep_tma).  The stage holds five planes: |kappa|, G, the static limit (field 2,
// or the override array), gh, and the forward velocities; the reciprocals of gh are made when the stage lands.  rec_w / vf_w / sb_w: block row 0 at the warp's
// LOWEST column; lc: this lane's column minus that one; o: sample lo of the final velocities (sample order).
template <int NT>
__device__ __forceinline__ void bwd_sweep_tma(const WarpRing& R, const double* __restrict__ rec_w, const double* __restrict__ vf_w,
                                              const double* __restrict__ sb_w, int lc, double* __restrict__ o, int lo, int len,
                                              double top_ak, double top_G, double top_st, const int* s_bi, const double* s_acc,
                                              int n_b, double acc0, double hw, double dd, double& v, double& sq, float& est,
                                              float dd_over_dt)
{
    constexpr int PD = TMA_PLANE_DOUBLES;
    const int lane = threadIdx.x & 31;
    const int nbl = (len + PB - 1) >> 2;                                      // block rows of this lane's chunk
    const int nbw = __reduce_max_sync(0xffffffffu, nbl);                      // block rows the warp streams (top down)
    if (lane == 0) {
        if (nbw > 0) ring_issue<NT>(R, 0, rec_w, vf_w, sb_w, nbw - 1);
        if (nbw > 1) ring_issue<NT>(R, 1, rec_w, vf_w, sb_w, nbw - 2);
    }
    int e = lo + len - 1;                            // current edge; the reference's loop index is i = e + 1
    int j = n_b - 1;
    double acc = acc0;
    while (j >= 0 && s_bi[j] > e + 1) { acc = s_acc[j]; j--; }
    int nb_next = (j >= 0) ? s_bi[j] : -1;
    double tak = top_ak, tG = top_G, tst = top_st;   // terms of sample e+1
#define BWD_T(ROW_)                                                                                                  \
        {                                                                                                            \
            const double gh_ = gh[ROW_], rg_ = rg[ROW_], f_ = S[4 * PD + ROW_];                                     \
            if (e + 1 == nb_next) { acc = s_acc[j]; j--; nb_next = (j >= 0) ? s_bi[j] : -1; }                         \
            const double vup = v;                                                                                    \
            v = bwd_step(tak, gh_, rg_, tst, pymin(f_, tG), v, sq, acc, hw, dd);                                     \
            est += t_est_term(vup, v, dd_over_dt);                                                                   \
            tak = S[ROW_]; tG = S[PD + ROW_]; tst = S[2 * PD + ROW_];                                                \
            --e;                                                                                                     \
        }
    const int nfull = len >> 2, rem = len & 3;
    o += nfull * PB;                                 // the ragged top block's samples
    for (int it = 0; it < nbw; ++it) {
        const int rb = nbw - 1 - it;                 // block row
        const int s = it & 1;
        mbar_wait(R.bar + 8 * s, (it >> 1) & 1);
        const double* S = R.stage + (size_t)s * 5 * PD + lc * PB;
        VAP_CHECK(7, lc >= 0 && lc < 32 && (unsigned)__cvta_generic_to_shared(S + 4 * PD + 3) + 8 <= R.smem_hi);
        double gh[PB], rg[PB];
#pragma unroll
        for (int r = 0; r < PB; r++) gh[r] = S[3 * PD + r];
#pragma unroll
        for (int r = 0; r < PB; r++) rg[r] = recip_for_pass(gh[r]);
        if (rb < nfull) {                            // a whole block of this lane's chunk: rows 3 .. 0
            o -= PB;
            BWD_T(3)
            const double v3 = v;
            BWD_T(2)
            const double v2 = v;
            BWD_T(1)
            const double v1 = v;
            BWD_T(0)
            st_d2(o, v, v1); st_d2(o + 2, v2, v3);   // the whole 32-byte sector
        } else if (rb == nfull && rem > 0) {         // ragged top of the path's last chunk: rows rem-1 .. 0
            if (rem > 2) { BWD_T(2) o[2] = v; }
            if (rem > 1) { BWD_T(1) o[1] = v; }
            BWD_T(0) o[0] = v;
        }
        __syncwarp();
        if (lane == 0 && it + 2 < nbw) ring_issue<NT>(R, s, rec_w, vf_w, sb_w, nbw - 3 - it);
    }
#undef BWD_T
}

struct BwdArgs {
    const double* p; const double* f; double* o; const double* sb; int lo, len; double top_ak, top_G, top_st;
    const int* s_bi; const double* s_acc; int n_b; double acc0, hw, dd; float dd_over_dt;
};
// cold, divergent code out of line (see fwd_rerun); st = {v, sq}
template <int NT, bool OVR>
__device__ __noinline__ bool bwd_rerun(const BwdArgs a, double* st, float* est, bool prev_same, double old_top)
{
    double v = st[0], sq = st[1];
    float e = *est;
    const bool merged = bwd_run<NT, RUN_RERUN, OVR>(a.p, a.f, a.o, a.sb, a.lo, a.len, a.top_ak, a.top_G, a.top_st, a.s_bi, a.s_acc,
                                                    a.n_b, a.acc0, a.hw, a.dd, v, sq, prev_same, e, a.dd_over_dt, old_top);
    st[0] = v; st[1] = sq; *est = e;
    return merged;
}
template <int NT, bool OVR>
__device__ __noinline__ void bwd_dry(const BwdArgs a, double* st)
{
    double v = st[0], sq = st[1];
    float e = 0.f;
    bwd_run<NT, RUN_DRY, OVR>(a.p, a.f, nullptr, a.sb, a.lo, a.len, a.top_ak, a.top_G, a.top_st, a.s_bi, a.s_acc, a.n_b, a.acc0,
                              a.hw, a.dd, v, sq, false, e, a.dd_over_dt);
    st[0] = v; st[1] = sq;
}

// Backward pass.  Thread k walks column nch-1-k (the k-th chunk counted from the end), so states flow from thread k-1 to
// thread k as in the forward kernel.  Reads the forward velocities (slot order) and writes the final ones straight into
// vel[B][D_cap] in sample order.  Also accumulates the travel-time estimate used to size the time-domain outputs.
template <int NT>
__global__ void __maxnreg__(VAP_PASS_REGS_TMA) k_bwd_chunked(
    const int* __restrict__ status, const double* __restrict__ cons, double dd, double dt, double end_vel,
    long long RS, long long D_cap, const int* __restrict__ n_samples, const double* __restrict__ rec, int E_cap,
    const double* __restrict__ max_accels, const int* __restrict__ bidx, const int* __restrict__ bval,
    const int* __restrict__ n_ev, const double* __restrict__ vfT, double* __restrict__ vel, float* __restrict__ t_est,
    int* __restrict__ rounds_out, int warm, int max_rounds, const double* __restrict__ statB, int ring_off)
{
    extern __shared__ __align__(128) unsigned char s_mem[];
    const int k = threadIdx.x;
    const long long b = blockIdx.x;
    double* s_endv = reinterpret_cast<double*>(s_mem);
    double* s_endw = s_endv + NT;
    double* s_usev = s_endw + NT;
    double* s_usew = s_usev + NT;
    double* s_acc = s_usew + NT;                                  // [E_cap] max_accels[bval[j] + 1] (applied at sample bidx[j])
    int* s_bi = reinterpret_cast<int*>(s_acc + E_cap);
    if (k == 0 && t_est) t_est[b] = 0.f;
    if (status[b] != ST_OK) return;
    const int D = n_samples[b];
    const int steps = D - 1;
    double* vo = vel + (size_t)b * D_cap;
    if (k == 0) { vo[D - 1] = end_vel; if (rounds_out) rounds_out[2 * b + 1] = 0; }
    if (steps <= 0) return;
    const int n_b = n_ev[2 * b + 1];
    for (int q = k; q < n_b; q += NT) {
        s_bi[q] = bidx[(size_t)b * E_cap + q];
        s_acc[q] = max_accels[(size_t)b * E_cap + bval[(size_t)b * E_cap + q] + 1];
    }
    const double acc0 = max_accels[(size_t)b * E_cap + bval[(size_t)b * E_cap + n_b - 1]];
    const int Lc = chunk_len(steps, NT);
    const int nch = (steps + Lc - 1) / Lc;
    const bool active = k < nch;
    const int col = active ? nch - 1 - k : 0;                      // column (forward chunk index)
    const int lo = col * Lc;
    const int len = (lo + Lc < steps) ? Lc : steps - lo;
    const double* P = rec + (size_t)b * RS * 4;
    const double* vf = vfT + (size_t)b * RS;
    const double hw = cons[b * 6 + 5] * 0.5;
    // with max_acceleration overrides the static limit of this pass is in statB (slot order, written by the pre-pass)
    const bool ovr = pass_has_override(max_accels + (size_t)b * E_cap, n_ev[2 * b], cons[b * 6 + 1]) != 0;
    const double* SB = statB + (size_t)b * RS;
    // every warp owns a two-stage ring (5 planes of 1 KB per stage) and two mbarriers behind the tables
    WarpRing R;
    constexpr int WARPS = (NT + 31) / 32;
    const int w = k >> 5;
    R.stage = reinterpret_cast<double*>(s_mem + ring_off) + (size_t)w * 2 * 5 * TMA_PLANE_DOUBLES;
    R.bar = (unsigned)__cvta_generic_to_shared(s_mem + ring_off + (size_t)WARPS * 2 * 5 * TMA_PLANE_DOUBLES * 8 + 16 * w);
    R.planes = 5;
    R.bytes = (NT < 32 ? NT : 32) * PB * 8;
#ifdef VAP_BOUNDS_CHECK
    R.rec_lo = P; R.rec_hi = P + 4 * RS; R.x_lo = vf; R.x_hi = vf + RS;
    R.smem_lo = (unsigned)__cvta_generic_to_shared(s_mem + ring_off);
    R.smem_hi = R.smem_lo + WARPS * 2 * 5 * TMA_PLANE_DOUBLES * 8;
    R.bar_hi = R.smem_hi + 16 * WARPS;
#endif
    if ((k & 31) == 0) { mbar_init(R.bar, 1); mbar_init(R.bar + 8, 1); fence_mbar_init(); }
    __syncthreads();

    auto rec_of = [&](int x, int fld) {                             // field fld (0-2) of sample x
        if (fld == 2 && ovr) return __ldg(SB + (x >= steps ? (int)(RS - 1) : edge_slot(x, Lc, NT)));
        if (x >= steps) return __ldg(P + 4 * RS - 3 + fld);
        const int cx = x / Lc, rx = x - cx * Lc;
        return __ldg(P + rec_index(rx, fld, cx, NT));
    };
    auto vf_at = [&](int x) { return vf[x >= steps ? (int)(RS - 1) : edge_slot(x, Lc, NT)]; };
    // terms of the sample above the chunk (sample lo+len): row 0 of the next column, or the tail
    double top_ak = 0.0, top_G = 0.0, top_st = 0.0;
    if (active) { top_ak = rec_of(lo + len, 0); top_G = rec_of(lo + len, 1); top_st = rec_of(lo + len, 2); }
    BwdArgs A;
    A.p = P + col * PB; A.f = vf + col * PB; A.o = vo + lo; A.sb = SB + col * PB; A.lo = lo; A.len = len;
    A.top_ak = top_ak; A.top_G = top_G; A.top_st = top_st; A.s_bi = s_bi; A.s_acc = s_acc; A.n_b = n_b; A.acc0 = acc0;
    A.hw = hw; A.dd = dd; A.dd_over_dt = (float)dd / (float)dt;
    float est = 0.f;                                  // travel-time estimate of this chunk's steps

    // ---- sweep 1: thread k > 0 may start `wl` steps ABOVE its chunk (in the next column) from the guess
    // v[s0] = min(vel_f[s0], G[s0+1]) (the state-independent part of what step s0+1 produces) and only compute until it
    // reaches its own range (see the forward kernel)
    {
        double v = end_vel, sq = 0.0;
        if (active) {
            if (k > 0) {
                const int hi = lo + len;                                   // sample at the top of this chunk (< D-1)
                const int len_up = (hi + Lc < steps) ? Lc : steps - hi;    // edges of the column above
                int wl = warm < len_up ? warm : len_up;
                if (hi + wl + 2 > D - 1) wl = (D - 1) - hi - 2 > 0 ? (D - 1) - hi - 2 : 0;
                wl &= ~(PB - 1);
                const int s0 = hi + wl;                                    // sample the guess is made at
                v = pymin(vf_at(s0), rec_of(s0 + 1, 1));
                double vp1 = end_vel;
                if (s0 + 2 <= D - 1) vp1 = pymin(vf_at(s0 + 1), rec_of(s0 + 2, 1));
                const double wp = vp1 * rec_of(s0 + 1, 0);
                sq = wp * wp;
                if (wl > 0) {
                    // edges s0-1 .. hi of column col+1 (rows wl-1 .. 0); the terms above the first of them are sample s0's
                    BwdArgs W = A;
                    W.p = P + (col + 1) * PB; W.f = vf + (col + 1) * PB; W.o = nullptr; W.sb = SB + (col + 1) * PB;
                    W.lo = hi; W.len = wl; W.top_ak = rec_of(s0, 0); W.top_G = rec_of(s0, 1); W.top_st = rec_of(s0, 2);
                    double st[2] = {v, sq};
                    if (ovr) bwd_dry<NT, true>(W, st); else bwd_dry<NT, false>(W, st);
                    v = st[0]; sq = st[1];
                }
            }
            s_usev[k] = v; s_usew[k] = sq;
            VAP_CHECK(5, col >= 0 && col * PB + PB <= PB * NT && (size_t)(((len + 3) >> 2) + 1) * 4 * PB * NT <= (size_t)(4 * RS - 3) &&
                             (size_t)(((len + 3) >> 2) + 1) * PB * NT <= (size_t)(RS - 1) && A.o + len <= vo + D - 1 &&
                             lo + len <= steps && D <= D_cap);
        }
        // the warp's columns: lane 0 has the highest (nch-1-32w); the ring holds the 32 columns that end there
        const int col_hi = nch - 1 - (k & ~31);
        const int cs = col_hi > 31 ? col_hi - 31 : 0;
        bwd_sweep_tma<NT>(R, P + cs * PB, vf + cs * PB, ovr ? SB + cs * PB : nullptr, active ? col - cs : 0, vo + lo, lo,
                          active ? len : 0, top_ak, top_G, top_st, s_bi, s_acc, n_b, acc0, hw, dd, v, sq, est, A.dd_over_dt);
        s_endv[k] = v; s_endw[k] = sq;
    }
    __syncthreads();

    // ---- fix-up rounds (states flow from thread k-1 to thread k, as in the forward kernel)
    int rounds = 0;
    for (int round = 1; round < NT && round <= max_rounds; round++) {
        bool need = false;
        double in_v = 0.0, in_w = 0.0;
        if (active && k >= round) {
            in_v = s_endv[k - 1]; in_w = s_endw[k - 1];
            need = !(same_bits(in_v, s_usev[k]) && same_bits(in_w, s_usew[k]));
        }
        if (!__syncthreads_or(need)) break;
        rounds = round;
        if (need) {
            double st[2] = {in_v, in_w};
            const bool ps = same_bits(in_v, s_usev[k]);
            const bool merged = ovr ? bwd_rerun<NT, true>(A, st, &est, ps, s_usev[k]) : bwd_rerun<NT, false>(A, st, &est, ps, s_usev[k]);
            s_usev[k] = in_v; s_usew[k] = in_w;
            if (!merged) { s_endv[k] = st[0]; s_endw[k] = st[1]; }
        }
        __syncthreads();
    }
    if (k == 0 && rounds_out) rounds_out[2 * b + 1] = rounds;

    // ---- travel-time estimate: the sum of the chunks' (single precision is plenty: it only sizes buffers)
    __syncthreads();
    float* s_f = reinterpret_cast<float*>(s_endv);      // end states are no longer needed
    s_f[k] = active ? est : 0.f;
    __syncthreads();
    if (k == 0 && t_est) {
        float tot = 0.f;
        for (int q = 0; q < NT; q++) tot += s_f[q];
        t_est[b] = tot;
    }
}

// slot order -> sample order (only the forward-only mode of vap_velocity_profile needs it: the backward pass writes sample
// order itself): vel[e] = vT[slot(e)], the last sample from slot RS-1.  One thread per sample.
__global__ void __launch_bounds__(256) k_untranspose(const int* __restrict__ status, const int* __restrict__ n_samples,
                                                     long long D_cap, long long RS, int NT,
                                                     const double* __restrict__ vT, double* __restrict__ vel,
                                                     unsigned tiles_x)
{
    const PathTile pt = path_tile(tiles_x);
    const long long b = pt.b;
    if (status[b] != ST_OK) return;
    const int D = n_samples[b];
    const int steps = D - 1;
    const int e = pt.x * blockDim.x + threadIdx.x;
    if (e >= D) return;
    const double* src = vT + (size_t)b * RS;
    const int Lc = steps > 0 ? chunk_len(steps, NT) : 1;
    vel[(size_t)b * D_cap + e] = (e < steps) ? src[edge_slot(e, Lc, NT)] : src[RS - 1];
}
