/*
 * vap.h -- C ABI of libvap.so, the B200 (sm_100a) batched spline -> motion-profile engine.
 *
 * The reference (RohitMovva/VexAutonomousPlanner) has no FFI layer: its boundary is the Python call
 * surface of src/splines and src/motion_profiling_v2.  Each entry point below replaces one function
 * of that surface (cited as file:line relative to the reference's src/) for a BATCH of independent
 * paths.  The Python mirror of the reference classes (vexautonomousplanner_b200/*.py) binds these
 * symbols with ctypes; INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; no C++ or torch types.
 *   - every pointer is a DEVICE pointer (caller-owned; e.g. torch.Tensor.data_ptr()) unless the
 *     parameter name starts with h_ (host).  Arrays are C-contiguous, path-major.
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, nothing synchronises.
 *   - return value: 0 on success, <0 on a launch/argument error (text via vap_last_error()).
 *     Per-path failures never abort the batch: they are reported in status[B]:
 *        0 ok | -1 reference returns False | -2 reference raises IndexError
 *        -3 reference raises ValueError    | -4 caller capacity too small: D_cap / T_cap, or a max_splines (Q_cap of the
 *           distance table) below the path's own spline count
 *        -5 the reference's time loop would not terminate for this input (e.g. max_dec >= 20 ft/s^2 makes a step
 *           move backwards) or would emit more than 5e7 rows: the engine stops instead of hanging the GPU
 *        -6 more node crossings / action-point candidates than the per-path event tables hold (N_max wraps,
 *           4 candidate samples per action point): a permanent condition, unlike -4 it does not go away on a retry.
 *           The time stage never returns it: a path whose position oscillates across an action point or a node
 *           (steps that move backwards, max_dec > 0.2 / dt) is redone there by the reference-shaped serial kernel.
 *   - the library keeps no global mutable state and allocates nothing.
 *
 * Packed layouts
 *   node_attr[B][N_max][12] f64 : x, y (feet), turn_deg, wait_time, max_velocity, max_acceleration,
 *                                 tangent_x, tangent_y, incoming_magnitude, outgoing_magnitude,
 *                                 rot_cos, rot_sin   (cos/sin of radians(turn)(+pi if reverse), evaluated
 *                                 on the host with numpy exactly as spline_manager.py:105-113 does)
 *   node_flags[B][N_max]   i32  : bit0 is_reverse_node, bit1 stop, bit2 tangent is not None
 *   n_nodes[B]             i32
 *   ap_attr[B][A_max][4]   f64  : t, wait_time, max_velocity, max_acceleration
 *   ap_flags[B][A_max]     i32  : bit1 stop
 *   n_ap[B]                i32
 *   cons[B][6]             f64  : max_vel, max_acc, max_dec, friction_coef, max_jerk, track_width
 *   seg[B][N_max-1][6][2]  f64  : rows p0, p1, d0, d1, dd0, dd1 of global segment g (node g -> g+1)
 *   first_node[B][N_max+1] i32  : node index at which spline k starts; entry S = N-1
 *   param_end[B][N_max]    f64  : spline.parameters[-1] per spline
 */
#ifndef VAP_H
#define VAP_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VAP_NODE_ATTRS 12
#define VAP_AP_ATTRS 4
#define VAP_FLAG_REVERSE 1
#define VAP_FLAG_STOP 2
#define VAP_FLAG_TANGENT 4

#define VAP_OK 0
#define VAP_ERR_FALSE (-1)
#define VAP_ERR_INDEX (-2)
#define VAP_ERR_VALUE (-3)
#define VAP_ERR_CAPACITY (-4)
#define VAP_ERR_DIVERGED (-5)
#define VAP_ERR_EVENTS (-6)

int vap_version(void);
const char* vap_last_error(void);

/* S0  QuinticHermiteSplineManager.build_path (spline_manager.py:42-172) + QuinticHermiteSpline.fit
 *     (quintic_hermite_spline.py:30-219,719-736).  scratch: f64 [B][N_max][9].  Optional (may be NULL):
 *     params[B][2*N_max]: every spline's `parameters` array, concatenated (N - 1 + S values);
 *     derivs[B][2*N_max][4]: first_derivatives / second_derivatives of every spline's control points.    */
int vap_build_path(int64_t B, int N_max, const double* node_attr, const int32_t* node_flags,
                   const int32_t* n_nodes, double* seg, int32_t* first_node, double* param_end,
                   double* seglen, int32_t* n_splines, int32_t* status, double* scratch, double* params,
                   double* derivs, void* stream);

/* S0' QuinticHermiteSpline.fit for stand-alone splines (quintic_hermite_spline.py:30-138): R runs of up to
 *     n_max control points.  xy[R][n_max][2]; tan_has[R][n_max] (i32 bit0: incoming set, bit1: outgoing set);
 *     tan_in/tan_out[R][n_max][2]; bnd[R][2][2] = starting / ending tangent; bnd_has[R]: bit0 / bit1 apply the
 *     starting / ending tangent to the segment table (a valid ndarray(2), :543-590), bit2 / bit3 the attribute
 *     "is not None" (what _compute_derivatives tests, :170,:181), bit4 use the caller's derivatives
 *     deriv_in[R][n_max][4] = (first.x, first.y, second.x, second.y) instead of computing them.
 *     Outputs seg[R][n_max-1][12], seglen[R][n_max], params[R][n_max], status[R], deriv_out[R][n_max][4] (or NULL).
 *     scratch: f64 [R][n_max][5].                                                                          */
int vap_fit_splines(int64_t R, int n_max, const int32_t* n_pts, const double* xy, const int32_t* tan_has,
                    const double* tan_in, const double* tan_out, const int32_t* bnd_has, const double* bnd,
                    double* seg, double* seglen, double* params, int32_t* status, double* scratch,
                    const double* deriv_in, double* deriv_out, void* stream);

/* Evaluation (get_point/derivative/second_derivative _at_parameter, spline_manager.py:204-275 ->
 * quintic_hermite_spline.py:221-251,473-541).  which: 0 point, 1 first, 2 second derivative,
 * 3 heading + curvature (Spline.get_heading/get_curvature, spline.py:48-80; out = {heading, curvature}).
 * n queries: path[q] selects the path, t[q] the global parameter; out[q][2].                           */
int vap_eval(int64_t n, const int32_t* path, const double* t, int which, int N_max, const double* seg,
             const int32_t* first_node, const double* param_end, const int32_t* n_splines, double* out,
             void* stream);

/* S1  build_lookup_table (spline_manager.py:426-475): samples per spline (reference default 1000).
 *     lut_d/lut_t[B][Q_cap] with Q_cap >= samples * max_b n_splines[b]; total_len[B].  status is in/out: a path with
 *     samples * n_splines[b] > Q_cap gets VAP_ERR_CAPACITY (and total_len 0), which every later stage skips.       */
int vap_build_lut(int64_t B, int N_max, const double* seg, const int32_t* first_node, const double* param_end,
                  const int32_t* n_splines, int32_t* status, int samples, int64_t Q_cap, double* lut_d,
                  double* lut_t, double* total_len, void* stream);
/* Optional accelerator of distance_to_time (spline_manager.py:291-318): an inverse index of the distance table, so that
 *     np.searchsorted(distances, d) is one seeded lookup plus a verification against the table instead of a 10-level
 *     binary search (identical result).  lut_inv[B][vap_lut_index_row_ints(Q_cap)] i32; pass it (or NULL) to
 *     vap_velocity_profile / vap_time_profile.                                                          */
int64_t vap_lut_index_row_ints(int64_t Q_cap);
int vap_build_lut_index(int64_t B, const int32_t* n_splines, const int32_t* status, int samples, int64_t Q_cap,
                        const double* lut_d, const double* total_len, int32_t* lut_inv, void* stream);

/* S2  precompute_path_properties (spline_manager.py:477-548): spn samples per node (default 1000).
 *     prop_k/prop_h[B][P_cap], P_cap >= spn * N_max.                                                   */
int vap_build_props(int64_t B, int N_max, const int32_t* n_nodes, const double* seg, const int32_t* first_node,
                    const double* param_end, const int32_t* n_splines, const int32_t* status, int spn,
                    int64_t P_cap, double* prop_k, double* prop_h, void* stream);

/* distance_to_time (spline_manager.py:291-318) and the snap gather _interpolate_property (:550-580) for
 * n queries.  what: 0 distance->t, 1 heading(t), 2 curvature(t).                                      */
int vap_query_tables(int64_t n, const int32_t* path, const double* x, int what, const int32_t* n_nodes,
                     const int32_t* n_splines, int samples, int64_t Q_cap, const double* lut_d,
                     const double* lut_t, const double* total_len, int spn, int64_t P_cap, const double* prop_k,
                     const double* prop_h, double* out, void* stream);

/* Accumulated distance grid d_0 = 0, d_{i+1} = fl(d_i + dd) (motion_profile_generator.py:91,122): identical
 * for every path with the same dd, so it is built once (single serial chain) and reused.              */
int vap_build_dgrid(int64_t n, double dd, double* dgrid, void* stream);

/* S3  forward_backward_pass, sampling loop (motion_profile_generator.py:112-176) without the event logic:
 *     n_samples[B] (= D), t/kap/th[B][D_cap].  status gets VAP_ERR_CAPACITY if D > D_cap.              */
int vap_dist_sample(int64_t B, const int32_t* n_nodes, const int32_t* n_splines, int32_t* status, int64_t n_grid,
                    const double* dgrid, int samples, int64_t Q_cap, const double* lut_d, const double* lut_t,
                    const double* total_len, int spn, int64_t P_cap, const double* prop_k, const double* prop_h,
                    int64_t D_cap, int32_t* n_samples, double* t, double* kap, double* th, void* stream);

/* S3 events + S4 forward pass + S5 backward pass (motion_profile_generator.py:93-176,188-314).
 *     vel[B][D_cap] out.  max_accels[B][E_cap], bidx/bval[B][E_cap], n_ev[B][2] (len(max_accels), len(map));
 *     E_cap >= N_max + A_max + 2.  t_est[B]: estimate of the number of time samples (for sizing S6).
 *     mode: 0 both passes, 1 forward only (for stage tests).                                           */
int vap_fwd_bwd(int64_t B, int N_max, int A_max, const double* node_attr, const int32_t* node_flags,
                const int32_t* n_nodes, const double* ap_attr, const int32_t* ap_flags, const int32_t* n_ap,
                const double* cons, const int32_t* status, double dd, double dt, double start_vel, double end_vel,
                int64_t D_cap, const int32_t* n_samples, const double* t, const double* kap, const double* th,
                double* vel, int E_cap, double* max_accels, int32_t* bidx, int32_t* bval, int32_t* n_ev,
                double* t_est, int mode, void* stream);

/* v2 of S3 + S4 + S5 in ONE call, the fast path that Engine.profile uses: same results, bit for bit, as vap_dist_sample
 *     + vap_fwd_bwd.  Distance sampling (motion_profile_generator.py:84-176) with sample-parallel event detection and a
 *     per-path replay of the sampling loop's event logic (:93-176), then the forward and backward passes (:188-314) with
 *     `chunks` speculative chunks per path that are re-run until they merge bitwise with the serial evaluation.
 *   The sampling fills a shared-memory tile from which a pre-pass hoists everything of a step that depends neither on
 *     the velocity state nor on the events (per sample |kappa|, the velocity caps, the static acceleration limit; per
 *     step the wheel-acceleration denominator; the passes make its reciprocal themselves), so kappa / theta per
 *     distance sample never go to memory: t / kap / th [B][D_cap] are inspection outputs (pass all three or three
 *     NULLs).  The static acceleration limits of paths with max_acceleration overrides are rewritten after the event
 *     resolution.
 *   n_samples[B] and status as in vap_dist_sample (status may also get VAP_ERR_EVENTS); max_accels[B][E_cap],
 *     bidx/bval[B][E_cap] and n_ev[B][2] as in vap_fwd_bwd, E_cap >= N_max + A_max + 2.  vr_idx/vr_val[B][E_cap]:
 *     the initial-velocity regimes, v0[i] = vr_val[j] for the last j with vr_idx[j] <= i; st_idx[B][E_cap]: the stop
 *     samples (initial velocity 0.01); n_vr[B][2]: the number of regimes and of stop samples.  ev_scratch: i32 scratch
 *     of vap_event_scratch_ints(B, N_max, A_max) elements.  ins_est[B] f32: rows the time stage will insert for waits /
 *     turn profiles (sizing only).
 *   The arrays the passes stream are chunk-interleaved in blocks of four steps (steps 4k .. 4k+3 of chunk c are one
 *     32-byte sector; sector (k, c) follows sector (k, c-1)) so that every warp-wide access is one contiguous run and a
 *     chunk re-run alone fetches only bytes it uses: rec [B][RS][4] f64 (per block four field planes of 4 x `chunks`
 *     doubles, 32 bytes per sample), statB / vel_f [B][RS] f64 (the backward pass's static acceleration limit, touched only for paths with
 *     max_acceleration overrides; forward velocities; both slot order), RS = vap_pass_row_slots(D_cap, chunks).
 *     chunks: a power of two from 8 to 256.
 *   vel[B][D_cap] (D_cap even): final velocities in sample order, written by the backward pass itself (mode 1: the
 *     forward velocities in sample order); t_est[B] f32: estimate of the number of time samples (for sizing S6);
 *     rounds[B][2]: fix-up sweeps of the forward / backward pass.  mode: 0 both passes, 1 forward only (stage tests). */
int64_t vap_event_scratch_ints(int64_t B, int N_max, int A_max);
int64_t vap_pass_row_slots(int64_t D_cap, int chunks);
int vap_velocity_profile(int64_t B, int N_max, int A_max, const double* node_attr, const int32_t* node_flags,
                         const int32_t* n_nodes, const double* ap_attr, const int32_t* ap_flags, const int32_t* n_ap,
                         const double* cons, const int32_t* n_splines, int32_t* status, int64_t n_grid,
                         const double* dgrid, int samples, int64_t Q_cap, const double* lut_d, const double* lut_t,
                         const double* total_len, int spn, int64_t P_cap, const double* prop_k, const double* prop_h,
                         const int32_t* lut_inv, double dd, double dt, double start_vel, double end_vel, int64_t D_cap,
                         int32_t* n_samples, double* t, double* kap, double* th, int E_cap, double* max_accels,
                         int32_t* bidx, int32_t* bval, int32_t* n_ev, int32_t* vr_idx, double* vr_val, int32_t* st_idx,
                         int32_t* n_vr, float* ins_est, int32_t* ev_scratch, double* rec, double* statB, double* vel_f,
                         double* vel, float* t_est, int32_t* rounds, int chunks, int mode, void* stream);

/* S6  generate_motion_profile time loop + node-0 prologue + turn / wait inserts
 *     (motion_profile_generator.py:414-628, one_dim_mp_generator.py:4-69) and S7 summary rows.
 *     out[8][B][T_cap]: times, positions, linear_vels, accelerations, headings, angular_vels, x, y.
 *     nodes_map[B][N_max+1] (with the caller's trailing len(times), gui/path.py:342), actions_map[B][A_max],
 *     n_maps[B][2]; n_out[B]; summary[B][5] = {n_out, total_length, t_end, max|v|, status}.
 *     If a path needs more than T_cap rows, n_out still holds the true count and status = -4.          */
int vap_resample(int64_t B, int N_max, int A_max, const double* node_attr, const int32_t* node_flags,
                 const int32_t* n_nodes, const double* ap_attr, const int32_t* ap_flags, const int32_t* n_ap,
                 const double* cons, int32_t* status, double dt, double dd, const double* seg,
                 const int32_t* first_node, const double* param_end, const int32_t* n_splines, int samples,
                 int64_t Q_cap, const double* lut_d, const double* lut_t, const double* total_len, int spn,
                 int64_t P_cap, const double* prop_k, const double* prop_h, int64_t D_cap,
                 const int32_t* n_samples, const double* vel, int64_t T_cap, double* out, int32_t* nodes_map,
                 int32_t* actions_map, int32_t* n_maps, int32_t* n_out, double* summary, void* stream);

/* v2 of S6 + S7 (same results, bit for bit, as vap_resample; this is the fast path).  The loop-carried state of
 *     the reference's time loop is only (current_pos, current_vel), so the stage runs as: the exact state recurrence
 *     (one thread per path), sample-parallel lookups + event candidates, a per-path replay of the event logic with the
 *     `current_time += dt` chain and the inserted rows, and a sample-parallel scatter to the final rows.
 *     D_cap must be a multiple of 128 (velocity rows are staged in 128-sample blocks through shared memory).
 *     n_main[B] i32: number of main-loop iterations (valid even on overflow); stage: f64 scratch [8][B][T_cap+1];
 *     seg_tab: i32 scratch [3*B*E_cap + B]; ev_scratch: i32 scratch of vap_event_scratch_ints elements.
 *     out_plane_stride: elements between the eight planes of `out` (0 = B*T_cap); lets a tile of a larger batch
 *     write straight into its rows of the batch-wide output.                                                   */
int vap_time_profile(int64_t B, int N_max, int A_max, const double* node_attr, const int32_t* node_flags,
                     const int32_t* n_nodes, const double* ap_attr, const int32_t* ap_flags, const int32_t* n_ap,
                     const double* cons, int32_t* status, double dt, double dd, const double* seg,
                     const int32_t* first_node, const double* param_end, const int32_t* n_splines, int samples,
                     int64_t Q_cap, const double* lut_d, const double* lut_t, const double* total_len, int spn,
                     int64_t P_cap, const double* prop_k, const double* prop_h, int64_t D_cap,
                     const int32_t* n_samples, const double* vel, int64_t T_cap, double* out, int32_t* nodes_map,
                     int32_t* actions_map, int32_t* n_maps, int32_t* n_out, double* summary, int32_t* n_main,
                     double* stage, int E_cap, int32_t* seg_tab, int32_t* ev_scratch, int64_t out_plane_stride,
                     const int32_t* lut_inv, const double* rden, int64_t n_rden, void* stream);
/* Optional accelerator of the time loop's lerp (motion_profile_generator.py:349-386 on xs[i] = i*dd, :484): rden[i] =
 *     1 / (xs[i+1] - xs[i]) for i < n, path-independent (depends on dd only).  With it the loop divides by one
 *     multiplication and two fused residual corrections (the IEEE quotient, bit for bit); pass NULL to divide directly. */
int vap_build_lerp_recip(int64_t n, double dd, double* rden, void* stream);

/* ---- The whole hot path behind ONE call ------------------------------------------------------------------------------
 * vap_profile_batch = build_path (spline_manager.py:42-172) + generate_motion_profile(spline_manager, constraints, dt, dd)
 * (motion_profile_generator.py:389-628, which starts with rebuild_tables, spline_manager.py:582) for B paths: S0 -> S7 on
 * `stream`, every intermediate carved out of ONE caller-owned workspace of vap_workspace_bytes(...) bytes (256-byte aligned;
 * the library allocates nothing).  The caller chooses the capacities: D_cap distance samples (a multiple of 128) and T_cap
 * time samples per path; sizing is checked on the device, per path: a path that needs more gets status VAP_ERR_CAPACITY
 * (its true counts are still in n_samples / n_out), the others are unaffected.  need[3] (device i64, may be NULL) receives
 * the batch maxima {distance samples, estimated time samples incl. inserted rows, a sufficient T_cap from the time loop's own
 * iteration count (0 while the distance samples did not fit)} over the paths that
 * are healthy or only lacked capacity: read it back to size a retry.  need[] does not report the spline count: a path with
 * more splines than max_splines also gets VAP_ERR_CAPACITY (n_samples = n_out = 0), and the caller finds the batch's true
 * count from vap_build_path's n_splines.  Paths whose length or travel time is absurd (the reference's loops would not
 * terminate) get VAP_ERR_DIVERGED.
 * Inputs: the packed node / action-point tables of vap_build_path / vap_velocity_profile; max_splines >= max_b n_splines[b]
 * (1 + the number of interior reverse / turn nodes; N_max - 1 is always enough; a smaller value gives VAP_ERR_CAPACITY on
 * exactly the paths that have more splines); dgrid[n_grid >= D_cap + 2] from vap_build_dgrid and
 * rden[n_rden] from vap_build_lerp_recip (or NULL): path-independent, depend on dd only, build them once.
 * Outputs: out[8][B][T_cap] (planes out_plane_stride elements apart, 0 = B*T_cap): times, positions, linear_vels,
 * accelerations, headings, angular_vels, x, y; n_out[B]; nodes_map[B][N_max+1]; actions_map[B][max(A_max,1)]; n_maps[B][2];
 * status[B]; summary[B][5]; vel[B][D_cap] (forward_backward_pass); n_samples[B].                                          */
int64_t vap_workspace_bytes(int64_t B, int N_max, int A_max, int max_splines, int lut_samples, int samples_per_node,
                            int64_t D_cap, int64_t T_cap, int chunks);
int vap_profile_batch(int64_t B, int N_max, int A_max, int max_splines, const double* node_attr,
                      const int32_t* node_flags, const int32_t* n_nodes, const double* ap_attr, const int32_t* ap_flags,
                      const int32_t* n_ap, const double* cons, double dt, double dd, double start_vel, double end_vel,
                      int lut_samples, int samples_per_node, int64_t D_cap, int64_t T_cap, int chunks, const double* dgrid,
                      int64_t n_grid, const double* rden, int64_t n_rden, void* workspace, int64_t workspace_bytes,
                      double* out, int64_t out_plane_stride, int32_t* n_out, int32_t* nodes_map, int32_t* actions_map,
                      int32_t* n_maps, int32_t* status, double* summary, double* vel, int32_t* n_samples, int64_t* need,
                      void* stream);
/* S7 on its own: summary[b] = {n_out, total_length (0 if total_len is NULL), times[-1], max |linear_vels|, status} from the
 * output streams (the rows the ranks of a sharded job gather).  vap_resample / vap_time_profile / vap_profile_batch already
 * write these rows; this entry serves callers that produced `out` some other way (a tile loop, a re-used buffer).        */
int vap_summary(int64_t B, int64_t T_cap, int64_t out_plane_stride, const double* out, const int32_t* n_out,
                const int32_t* status, const double* total_len, double* summary, void* stream);

/* S1' QuinticHermiteSpline.get_arc_length (Gauss-Legendre, quintic_hermite_spline.py:592-644) and
 *     get_parameter_by_arc_length (:661-717) for n queries on spline `spl[q]` of path `path[q]`.
 *     gl_pts / gl_wts[npts] = np.polynomial.legendre.leggauss(npts) from the host (device copies).
 *     mode 0: out[q] = arc length over [a[q], b[q]]; mode 1: out[q] = parameter at arc length a[q]
 *     (b[q] = tolerance, max_iter iterations).  qstatus[q] = 0 or VAP_ERR_VALUE.                       */
int vap_gl(int64_t n, const int32_t* path, const int32_t* spl, const double* a, const double* b, int mode,
           int max_iter, int npts, const double* gl_pts, const double* gl_wts, int N_max, const double* seg,
           const int32_t* first_node, const double* param_end, double* out, int32_t* qstatus, void* stream);

/* motion_profile_angle (motion_profile_generator.py:319-346) / generate_trapezoidal_profile
 * (one_dim_mp_generator.py:4-69) for n queries: q[n][5] = angle_rad (or total_distance when mode 1),
 * max_vel, max_acc, track_width, dt.  mode 0: out_a = headings, out_b = angular velocities;
 * mode 1: out_a = velocities.  Rows of K_cap; counts[n].                                               */
int vap_turn_profile(int64_t n, const double* q, int mode, int64_t K_cap, double* out_a, double* out_b,
                     int32_t* counts, void* stream);

/* lerp (motion_profile_generator.py:349-386, cache=None) of n queries against one sorted table xs/ys[m],
 * and get_wheel_trajectory (:631-646).                                                                  */
int vap_lerp(int64_t n, const double* x, int64_t m, const double* xs, const double* ys, double* out, void* stream);
int vap_wheel_trajectory(int64_t n, const double* lin, const double* ang, double track_width, double* left,
                         double* right, void* stream);

/* Dense packing of the result rows: offsets[B+1] (i64) = exclusive prefix sum of min(n_out, T_cap) over the ok paths,
 * dst[8*offsets[b] + s*n_b + k] = out[s][b][k] for the eight planes s.  `dst` may be pinned (mapped) HOST memory: the
 * kernel then streams exactly the valid rows over PCIe, which is how the Python layer returns results to the host
 * (the reference hands back Python lists, motion_profile_generator.py:618-628).                                  */
int vap_pack_rows(int64_t B, int64_t T_cap, int64_t out_plane_stride, const double* out, const int32_t* n_out,
                  const int32_t* status, int64_t* offsets, double* dst, void* stream);

/* "Next" row f1: numeric rows of the trajectory export written by save_nodes_to_file (gui_manager.py:284-295):
 * dst[7*(offsets[b] + k) + {0..6}] = {0, t, x*12, y*-12, heading, v*12, omega} for every time sample k of path b;
 * offsets[B+1] as in vap_pack_rows.  Their text is produced by vap_format_rows below; the handful of action rows
 * ([1, *action_values], :297-310) is spliced on the host (vexautonomousplanner_b200/export.py).                 */
int vap_export_rows(int64_t B, int64_t T_cap, int64_t out_plane_stride, const double* out, const int32_t* n_out,
                    const int32_t* status, int64_t* offsets, double* dst, void* stream);

/* "Next" row f1, text: Python's repr(float) (= what f"{v} " writes, gui_manager.py:220-230) on the device.
 *   vap_format_doubles: n values -> 32-byte NUL-padded slots out32[n][32] + lens[n].
 *   vap_format_rows: export rows[R][7] -> one line per row ("0 t x y heading v omega \n", every value followed by a
 *     blank) in slots[R][vap_row_text_stride()] + lens[R]; kinds[R] (u8 bit set from vap_row_kinds, may be NULL) prints
 *     the columns that hold a Python int in the reference as "0" instead of "0.0".  vap_compact_rows then copies line r
 *     to text + offsets[r] (offsets[R] i64: the byte position of line r; the exclusive prefix sum of lens gives one
 *     contiguous text buffer, the line_dst of vap_splice_plan leaves the gaps for the action rows).
 *   vap_row_kinds: per result row of every path, which entries of generate_motion_profile's lists are Python ints
 *     (motion_profile_generator.py:425, 448-453, 459-476, 487-518, 548-553): bit 1 times[r] (row 0 without a prologue),
 *     bit 2 linear_vels / accelerations (inserted turn / wait rows), bit 4 angular_vels (wait rows, first turn row),
 *     bit 8 positions (wait rows).  kinds row of path b starts at offsets[b] (the dense rows of vap_export_rows) or at
 *     b * T_cap when offsets is NULL; n_kinds = bytes of `kinds` (cleared by the call).                            */
int vap_row_kinds(int64_t B, int N_max, int A_max, const double* node_attr, const int32_t* n_nodes, const double* ap_attr,
                  const int32_t* n_ap, const double* cons, const int32_t* status, double dt, const int32_t* nodes_map,
                  const int32_t* actions_map, const int32_t* n_maps, const int32_t* n_out, int64_t T_cap,
                  const int64_t* offsets, int64_t n_kinds, uint8_t* kinds, void* stream);
int vap_format_doubles(int64_t n, const double* x, char* out32, int32_t* lens, void* stream);
int vap_row_text_stride(void);
int vap_format_rows(int64_t R, const double* rows, const uint8_t* kinds, char* slots, int32_t* lens, void* stream);
int vap_compact_rows(int64_t R, const char* slots, const int32_t* lens, const int64_t* offsets, char* text, void* stream);

/* "Next" row f1, the whole .txt body of every path (save_nodes_to_file, gui_manager.py:284-316): the path's trajectory
 * lines with the action rows inserted as the reference does it, list.insert(nodes_map[i] + i, row) for i < n_maps[b][0],
 * then list.insert(actions_map[j] + j, row) for j < n_maps[b][1] (Python's clamping: an index past the end appends, a
 * negative one counts from the end and stops at 0; the action-point indices do not count the node rows before them).
 *   vap_splice_plan: the lines of path b are the dense rows row_offsets[b] .. row_offsets[b+1] of vap_export_rows;
 *     line_offsets[R+1] (i64) = exclusive prefix sum of the line lengths of vap_format_rows (R = row_offsets[B]).  The
 *     action rows are caller text (the host formats [1, *action_values] with f"{v} "): act_text[act_off[i] .. act_off[i+1])
 *     is row i of n_act, act_off[n_act+1] i64; the rows of path b start at act_first[b] (i64), its act_rows[b][0] node
 *     rows first, then its act_rows[b][1] action-point rows.  nodes_map / actions_map / n_maps as vap_time_profile writes
 *     them (rows of N_max + 1 and max(A_max, 1) entries).
 *     Outputs: path_offsets[B+1] (i64): path b's body is text[path_offsets[b] .. path_offsets[b+1]); line_dst[R] (i64): byte
 *     position of every trajectory line, for vap_compact_rows; act_dst[n_act] (i64): byte position of every action row,
 *     -1 for rows that are in no body; flags[B] (i32): 0 assembled, 1 status[b] != 0 (no action rows; vap_export_rows
 *     gives such a path no lines either, so its body is empty), 2 the maps need more
 *     rows than act_rows passes (or n_maps exceeds the map rows): nothing of the action rows is read, the body holds
 *     the trajectory lines only.  Read path_offsets[B] back to size `text`.  Shared memory per path:
 *     32 * (N_max + 1 + max(A_max, 1)) bytes.
 *   vap_splice_actions: copies row i of act_text to text + act_dst[i] (after vap_compact_rows with line_dst, or before).  */
int vap_splice_plan(int64_t B, int N_max, int A_max, const int32_t* status, const int32_t* nodes_map,
                    const int32_t* actions_map, const int32_t* n_maps, const int64_t* row_offsets,
                    const int64_t* line_offsets, const int64_t* act_first, const int32_t* act_rows, int64_t n_act,
                    const int64_t* act_off, int64_t* path_offsets, int64_t* line_dst, int64_t* act_dst, int32_t* flags,
                    void* stream);
int vap_splice_actions(int64_t n_act, const char* act_text, const int64_t* act_off, const int64_t* act_dst, char* text,
                       void* stream);

/* "Next" row f1 read back: the text of saved .txt bodies on the device.  A token is [-]digits[.digits][e[+|-]digits],
 * [-]inf or [-]nan; its value is bit-equal to Python's float(token) (Clinger's fast path, then Eisel-Lemire with a
 * 128-bit truncated 5^q).  A token the device does not decide (more than 19 significant digits whose rounding the
 * digits kept cannot settle, or an ambiguous 128-bit product) is left to the caller's float(), never guessed.
 *   vap_parse_doubles: token i = text[tok_off[i] .. tok_off[i+1]) (tok_off[n+1] i64) -> out[i] and flags[i] (i8): 0 parsed,
 *     1 left for float() (out NaN), 2 not a token of the grammar (out NaN).                                          */
int vap_parse_doubles(int64_t n, const char* text, const int64_t* tok_off, double* out, int8_t* flags, void* stream);

/* Lines of B bodies concatenated in one buffer: body b is text[path_off[b] .. path_off[b+1]) (path_off[B+1] i64,
 * path_off[B] = n_bytes).  A line ends after '\n' or at the end of its body.  Four calls, the caller scanning between:
 *   vap_line_starts: starts[n_bytes] (u8) = 1 where a line starts.
 *   vap_line_offsets: scan[n_bytes] (i32) = inclusive prefix sum of starts; L = scan[n_bytes - 1] lines.  Writes
 *     line_off[L+1] (i64, line_off[L] = n_bytes) and path_line_off[B+1] (i64): body b owns lines path_line_off[b] ..
 *     path_line_off[b+1].
 *   vap_line_kinds: kinds[L] (u8) 0 trajectory row (first token "0"), 1 action row (first token "1"), 2 other;
 *     errors[L] (i32) 0, 1 blank line, 2 first token neither 0 nor 1; counts[L] (i64) = (kind == 0) + 2^32 (kind == 1).
 *   vap_parse_rows: count_scan[L] (i64) = inclusive prefix sum of counts (both running counts at once).  Writes path_row_off[B+1]
 *     and path_act_off[B+1] (i64): body b owns trajectory rows path_row_off[b] .. and action rows path_act_off[b] ..;
 *     act_line[] (i64, one per action row) = its line; for the trajectory rows of the first parse_paths bodies
 *     rows[r][7] = {0, t, x, y, heading, v, omega} as written, host_mask[l] (u8, cleared by the call) bit c = token c of
 *     line l left for float(), errors[l] = 3 when the row has not exactly 7 tokens, 4 + c when token c is not a token
 *     of the grammar.  rows, act_line: at most L entries.                                                          */
int vap_line_starts(int64_t B, int64_t n_bytes, const char* text, const int64_t* path_off, uint8_t* starts, void* stream);
int vap_line_offsets(int64_t B, int64_t n_bytes, const uint8_t* starts, const int32_t* scan, const int64_t* path_off,
                     int64_t* line_off, int64_t* path_line_off, void* stream);
int vap_line_kinds(int64_t L, const char* text, const int64_t* line_off, uint8_t* kinds, int32_t* errors, int64_t* counts,
                   void* stream);
int vap_parse_rows(int64_t B, int64_t L, const char* text, const int64_t* line_off, const uint8_t* kinds,
                   const int64_t* count_scan, const int64_t* path_line_off, int64_t parse_paths, int64_t* path_row_off,
                   int64_t* path_act_off, int64_t* act_line, double* rows, uint8_t* host_mask, int32_t* errors, void* stream);

/* A saved body against a fresh one, per path b (one warp each): saved body text[old_off[b] .. old_off[b+1]), fresh body
 * text[new_off[b] .. new_off[b+1]) (the same buffer, e.g. both sets split by the calls above with 2B bodies).  line_off,
 * line_err, act_line as above; the saved body's lines start at old_path_line_off[b]; the saved and fresh action rows of
 * b start at old_path_act_off[b] / new_path_act_off[b] in act_line; old_rows / new_rows [.][7] with their per-path row
 * offsets (the parsed rows, and the rows of vap_export_rows).
 *   out_i64[B][7]: first differing byte from the body start (-1 equal), its line in the saved body from 1 (0 equal),
 *     saved and fresh trajectory rows, action rows that differ (the k-th saved against the k-th fresh; unpaired ones
 *     count), first saved line with an error from 1 (0 none), its error code.
 *   out_f64[B][8]: t of the last saved and of the last fresh row (NaN without rows), max |saved - fresh| of t, x, y,
 *     heading, v, omega over the common rows (row k against row k; inf where exactly one is NaN).                  */
int vap_compare_bodies(int64_t B, const char* text, const int64_t* old_off, const int64_t* new_off, const int64_t* line_off,
                       const int32_t* line_err, const int64_t* old_path_line_off, const int64_t* act_line,
                       const int64_t* old_path_act_off, const int64_t* new_path_act_off, const double* old_rows,
                       const int64_t* old_row_off, const double* new_rows, const int64_t* new_row_off, int64_t* out_i64,
                       double* out_f64, void* stream);

/* The robot's rectangle along the export rows, per path b (one CTA each): rows[R][7] = {0, t, x, y, heading, v, omega}
 * (inches, heading CCW from +x), path b owning rows row_off[b] .. row_off[b+1] (row_off[B+1] i64: vap_export_rows, or
 * the rows vap_parse_rows read back).  The rectangle is centred on (x, y), hl inches to the front and back along the
 * heading, hw inches to each side; the field is xmin..xmax by ymin..ymax; boxes (HOST memory, K <= 64) [K][4] =
 * {x0, y0, x1, y1} are axis-aligned keep-out boxes.  Per row: wall margin = largest overhang of a corner past a field
 * edge (negative: clearance), box distance = Euclidean distance between the rectangles, or minus the penetration depth
 * (the smallest overlap of the four separating axes) when they overlap.  A row violates when its wall margin > tol, a
 * box distance < -tol, or x, y or heading is not finite.  Row numbers count from 0 within the path; ties go to the
 * lowest row, then the lowest box.
 *   out_i64[B][7]: rows, first violating row (-1 none), its kind (-1 none, 0 wall, 1 not finite, 2 + k box k), number
 *     of violating rows, row of the largest wall margin, row of the smallest box distance and that box (-1 / -1 when
 *     K = 0; -1 everywhere without a finite row).
 *   out_f64[B][6]: t of the first violation (NaN none), largest wall margin (-inf without a finite row) and its t,
 *     smallest box distance (+inf when K = 0) and its t, largest displacement of a corner between consecutive finite
 *     rows (what sampling can miss between two rows).
 * Returns < 0 with vap_last_error for hl or hw not positive, an empty field box, K outside 0..64, an empty box, or a
 * tolerance that is not finite.                                                                                    */
int vap_footprint_check(int64_t B, const double* rows, const int64_t* row_off, double hl, double hw, double xmin, double xmax,
                        double ymin, double ymax, int K, const double* boxes, double tol, int64_t* out_i64, double* out_f64,
                        void* stream);

/* Bounds diagnostics of a -DVAP_BOUNDS_CHECK build (profiles/tools/bounds_check.py; compute-sanitizer is closed on the GPU
 * pool this was developed on): out_host[32] (HOST memory) = violations per check site (0..15) and checks executed per site
 * (16..31); returns <0 in a release build, where the checks are compiled away.                                          */
int vap_diag_read(uint64_t* out_host, int reset);

/* Measurement hook: `ctas` CTAs of 256 threads run `iters` rounds of 8 independent fp64 FMA chains each
 * (flops = ctas * 256 * iters * 16); bench.py times it to report the MEASURED fp64 peak that fp64-pipe
 * utilisations are quoted against (BASELINE.md section 3).  out: one device double (never written).        */
int vap_bench_dfma(int64_t ctas, int64_t iters, double* out, void* stream);

/* Test hook: counts (into the device word *bad) the pseudo-random numerators a, out of n, for which the hoisted-
 * reciprocal division used inside the time loop differs from the IEEE quotient a / b.  Must stay 0.            */
int vap_test_div_const(int64_t n, uint64_t seed, double b, uint64_t* bad, void* stream);
/* test hook: mismatches between the velocity passes' pre-computed-reciprocal division and IEEE '/' over n random pairs */
int vap_test_div_recip(int64_t n, uint64_t seed, uint64_t* bad, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VAP_H */
