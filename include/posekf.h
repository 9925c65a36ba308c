/* posekf.h -- C ABI of libposekf_b200.so: the B200 (sm_100a) batched quaternion EKF.
 *
 * This is the drop-in boundary for the offline replay path of varunbachalli/PoseEstimationKF.
 * The reference has no FFI layer for this path -- its boundary is the Python import surface used by
 * `Python Kalman Filter/main_file.py:1-6` -- so every entry point below cites the reference
 * Python function (file:line, relative to the reference repository; PKF = "Python Kalman Filter",
 * SRV = "Kalman Filter Server/PoseEstimator") whose arithmetic it replaces for a batch of N
 * independent filters.  INTEGRATION.md shows the ctypes binding a maintainer of the reference adds.
 *
 * Conventions
 *   - All pointers are DEVICE pointers unless the function name ends in `_host`.
 *   - Batched arrays are component-major ("structure of arrays"): a per-filter k-vector is stored
 *     as float[k][N] so that consecutive filters are consecutive in memory (coalesced).
 *     Matrices are row-major flattened: a 4x4 is float[16][N], entry (i,j) at row 4*i+j.
 *   - Quaternions are scalar-first [w,x,y,z]  (PKF/ExtendedKalmanFilter.py:17, PKF/Wahba.py:47).
 *   - Kernels never allocate or free; outputs are caller-allocated.  No global state: every entry
 *     point is re-entrant.  Launches are asynchronous on `stream` (a cudaStream_t, may be NULL).
 *   - Return value: 0 = ok; >0 = a cudaError_t; <0 = invalid argument (POSEKF_EINVAL...).
 *   - NaN/Inf propagate as in the reference (nothing is clamped silently).
 */
#ifndef POSEKF_H_
#define POSEKF_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define POSEKF_EINVAL (-1)      /* bad size / null pointer / bad enum                     */
#define POSEKF_EALIGN (-2)      /* pointer or stride alignment requirement not met        */
#define POSEKF_ENODEV (-3)      /* no sm_100 device / driver entry point unavailable      */

/* Wahba solver selection (see DESIGN.md "Wahba stage") */
#define POSEKF_WAHBA_QR2    0   /* rank-2 forms that never build B: stand-alone entry points use the QR of both vector
                                   pairs + closed-form 2x2 polar factor; the fused replay solves for the quaternion
                                   directly (two-observation closed form) and keeps the former for negative weights */
#define POSEKF_WAHBA_JACOBI 1   /* the SVD of PKF/Wahba.py:14 as a one-sided (Hestenes) Jacobi SVD in registers, QR-preconditioned:
                                   B = ka r_a a^T + km r_m m^T has rank 2, so the rotation is applied to its 2x2 core
                                   (QR of both vector pairs, heavier pair first); accurate to float32 rounding for any
                                   weights, including the reference's near-rank-1 (|a_z|, 1-|a_z|).  One thread per problem */
#define POSEKF_WAHBA_PRECOMPUTED 2 /* posekf_replay_f32 only: stream rows 3-6 already hold the Wahba quaternion
                                      (posekf_measurement_stream_f32) -- for (Q,R) sweeps over shared streams */

/* Stream staging selection for posekf_replay_f32 */
#define POSEKF_STAGE_AUTO 0     /* TMA when alignment allows, else LDG */
#define POSEKF_STAGE_LDG  1     /* coalesced global loads, register prefetch one step ahead */
#define POSEKF_STAGE_TMA  2     /* cp.async.bulk.tensor (TMA) multi-stage shared-memory ring */
#define POSEKF_STAGE_TMA_PACKED 3 /* same ring, two filters per thread in packed f32x2 registers (FFMA2);
                                     rank-2 Wahba, N even; what AUTO picks when eligible */

/* State frame flags of posekf_replay_f32 (bit mask).  The kernels run the filter in the coordinates of the
 * reference frame E = [e1 e2 e3] built from (acc_0, mag_0) -- the recursion is equivariant under a fixed
 * left rotation of the state, and in that frame the Wahba stage loses its 3x3 matrix product.  By default
 * (0) state_x / state_x_lo / state_p are read and written in the reference's own coordinates and converted
 * at both ends of the launch.  A caller that replays in time chunks sets OUT on every launch but the last
 * and IN on every launch but the first: the state then stays in the filter frame between launches and the
 * chunked replay equals the unchunked one bit for bit (checkpoint / resume).  A launch with n_steps = 0
 * and exactly one flag set only converts the state.  Ignored by POSEKF_WAHBA_PRECOMPUTED launches, whose
 * filter frame is the reference frame. */
#define POSEKF_STATE_IN_FILTER_FRAME  1
#define POSEKF_STATE_OUT_FILTER_FRAME 2

/* Library / build info: returns a static string such as "posekf_b200 0.2 sm_100a". */
const char* posekf_version(void);

/* ---------------------------------------------------------------------------------------------
 * Fused replay: T steps of Prediction+Correction for N filters in one launch.
 * Replaces the loop body of PKF/main_file.py:38-47, i.e. per step and filter
 *   KalmanFilter.Prediction  PKF/ExtendedKalmanFilter.py:58-68  (GetJacobian_A :43-48,
 *                            GetJacobian_B :51-56, RungeKutta4 :25-41, inv :65)
 *   KalmanFilter.Correction  PKF/ExtendedKalmanFilter.py:70-80  (Wahba.getQuarternion
 *                            PKF/Wahba.py:49-50 -> getRotation :8-17, RotationMatrix2Quart :20-47,
 *                            Comparator :16-23, norm PKF/UtilityFunctions.py:16-21)
 * and optionally the accel/mag low-pass of SRV/KalmanFilter.cpp:21-24 (PKF/Test.py:27-33).
 *
 *   n_filters   N
 *   n_steps     T
 *   streams     [T][9][Ns] : rows 0-2 gyro (rad/s), 3-5 acc, 6-8 mag
 *   n_streams   Ns: number of distinct input columns; filter n reads column n % Ns.  Ns == N for a
 *               plain replay; Ns < N (N % Ns == 0) for a Q/R sweep that shares trajectories.
 *   dt          seconds between samples: one float (dt_per_step = 0) or [T] (dt_per_step = 1).
 *               (The reference passes integer ns timestamps and differences them,
 *               PKF/ExtendedKalmanFilter.py:32,62; ns do not fit float32, so the caller differences.)
 *   acc_ref, mag_ref  [3][Ns] : the log's acc_0 / mag_0 (Wahba reference vectors, PKF/Wahba.py:4-6)
 *   q_scale, r_scale  [N] : Q = q*I3, R = r*I4 as produced by setQ/setR (PKF/ExtendedKalmanFilter.py:12-15);
 *               r must be > 0 (the kernel carries the covariance in units of r), q >= 0
 *   lpf_alpha_acc/mag  low-pass coefficient, < 0 disables the stage
 *   state_x     [4][N]  in: X before the first step, out: X after the last step
 *   state_x_lo  [4][N] in/out or NULL.  Non-NULL selects the PRECISE variant for extreme Q/R ratios: X is
 *               carried as two floats (state_x + state_x_lo) so that corrections below half an ulp of the
 *               state are not lost (R >> Q: 2.4e-5 rad from the reference after 5000 steps at Q=1e-3,
 *               R=1e3 otherwise), and the gain is formed by Sherman-Morrison with the process noise kept
 *               apart from A K A^T (Q >> R: 1.7e-5 rad spikes at Q=1e3, R=1e-3 otherwise).  <= 3.5e-7 rad over
 *               the whole 1e-3..1e3 grid; costs ~25 % more time.  Start at 0.
 *               VALIDITY OF THE PLAIN VARIANT (NULL): 1e-2 < q/r < 1e4 for every filter.  Outside that range it
 *               leaves the 1e-5 rad tolerance -- quickly for r >> q, where the diagonal of its gain, formed as
 *               1 - 1/d, cancels (3e-3 rad at q/r = 1e-6).  Device pointers cannot be checked here: the Python layer
 *               selects the variant from the values and refuses the plain one outside its range.
 *   state_p     [10][N] in/out: upper triangle of P / r  (the covariance IN UNITS OF THE FILTER'S r; after
 *               an update this equals the Kalman gain) in the order 00 01 02 03 11 12 13 22 23 33.
 *               The kernel works in this scaled form, so storing it unscaled would make a chunked
 *               replay differ from an unchunked one by an ulp; callers multiply by r to obtain P.
 *   state_lpf   [6][N]  in/out low-pass state (acc xyz, mag xyz); may be NULL when both alphas < 0
 *   out_traj    [T][N][4] state after every step (one 16-byte quaternion per filter-step, i.e. the
 *               reference's X_k list, PKF/main_file.py:44, for every filter), 16-byte aligned, or NULL
 *   out_flip    [T][N] uint8, 1 where the comparator negated the Wahba quaternion
 *               (PKF/ExtendedKalmanFilter.py:73-75), or NULL.  With POSEKF_WAHBA_QR2 on raw samples (no low-pass) the
 *               mask is the float64 reference's bit for bit: steps where its 3-branch sign rule (PKF/Wahba.py:26-47)
 *               sits on a float32 tie are re-decided in float64 by a second small kernel launched by this call
 *   truth       [T][Ns][4] reference track (ground truth, a Wahba-only or gyro-only track, another
 *               run's out_traj ...) for the on-device tuning objective, 16-byte aligned, or NULL
 *   loss_acc    [N] in/out, required with truth: loss_acc[n] += sum_t |X_t ^ truth_t|^2 = 1 - (X_t . truth_t)^2
 *               (sin^2 of the quaternion angle, evaluated as the squared wedge product).  Lets a Q/R sweep return its loss surface without storing
 *               trajectories (the tuning workflow of the reference's README, knobs main_file.py:21-22).
 *   wahba_algo  POSEKF_WAHBA_*
 *   staging     POSEKF_STAGE_*
 *   state_flags POSEKF_STATE_*_FILTER_FRAME bit mask, 0 = state in the reference's coordinates on both sides
 */
int posekf_replay_f32(int64_t n_filters, int64_t n_steps, const float* streams, int64_t n_streams,
                      const float* dt, int dt_per_step, const float* acc_ref, const float* mag_ref,
                      const float* q_scale, const float* r_scale, float lpf_alpha_acc, float lpf_alpha_mag,
                      float* state_x, float* state_x_lo, float* state_p, float* state_lpf, float* out_traj,
                      uint8_t* out_flip, const float* truth, float* loss_acc, int wahba_algo, int staging,
                      int state_flags, void* stream);

/* The same replay with the INNOVATION LIKELIHOOD of every filter accumulated on the device: a (Q,R) tuning objective
 * that needs no ground truth (a recorded log has none).  It is the filter's own Gaussian model of its innovations
 * (prediction-error decomposition), natural log, P and R unscaled:
 *     l(Q,R) = 1/2 sum_t [ NIS_t + ln det S_t + 4 ln 2 pi ],   NIS_t = e_t^T S_t^-1 e_t,
 *     S_t = P_t + R   (the matrix inverted at PKF/ExtendedKalmanFilter.py:63-65),
 *     e_t = y_t - z_t (the innovation of :76, y sign-fixed by the comparator :73-75).
 * All parameters are those of posekf_replay_f32, plus
 *   innov_acc   [2][N] in/out, required (NULL: POSEKF_EINVAL), 4-byte aligned (8-byte for the packed kernel; AUTO
 *               falls back to the scalar TMA kernel otherwise):  innov_acc[0][n] += sum_t NIS_t,
 *               innov_acc[1][n] += sum_t ln det S_t over the n_steps of the launch.  Start at 0 and pass the same buffer
 *               to every launch of a time-chunked replay (with the state flags above): the sums equal the unchunked
 *               replay's bit for bit.  Then  NLL = (innov_acc[0] + innov_acc[1]) / 2 + 2 T ln 2 pi,
 *               mean NIS = innov_acc[0] / T.
 * The statistic does not perturb the filter: state, trajectory and flip mask are those of posekf_replay_f32.  Both
 * terms are invariant under the kernels' filter-frame rotation.  Combinations of the packed staging with per-step
 * outputs or the low-pass run in the scalar kernels (same results bit for bit). */
int posekf_replay_innovation_f32(int64_t n_filters, int64_t n_steps, const float* streams, int64_t n_streams,
                                 const float* dt, int dt_per_step, const float* acc_ref, const float* mag_ref,
                                 const float* q_scale, const float* r_scale, float lpf_alpha_acc, float lpf_alpha_mag,
                                 float* state_x, float* state_x_lo, float* state_p, float* state_lpf, float* out_traj,
                                 uint8_t* out_flip, const float* truth, float* loss_acc, float* innov_acc, int wahba_algo,
                                 int staging, int state_flags, void* stream);

/* Which innovation likelihood posekf_replay_innovation_ex_f32 accumulates. */
#define POSEKF_INNOV_FULL    0  /* the 4-D model above: the sums of posekf_replay_innovation_f32, bit for bit */
#define POSEKF_INNOV_TANGENT 1  /* the same model in the 3-D tangent space of the prediction (below) */

/* posekf_replay_innovation_f32 with a choice of model.  POSEKF_INNOV_TANGENT leaves out the direction of the
 * prediction u_t = z_t/|z_t|: y and z are unit quaternions, so e.u ~ -|e|^2/2 carries almost no information, and P_t
 * leaves that direction almost empty, which makes the 4-D likelihood favour ever smaller R.  With E_t any 4x3
 * orthonormal basis of u_t-perp (the result does not depend on the choice):
 *     l_3(Q,R) = 1/2 sum_t [ NIS3_t + ln det S3_t + 3 ln 2 pi ],   S3_t = E_t^T S_t E_t,   e3_t = E_t^T e_t,
 *     NIS3_t = e3_t^T S3_t^-1 e3_t.
 *   innov_acc[0][n] += sum_t NIS3_t, innov_acc[1][n] += sum_t ln det S3_t; layout, alignment, chunking and routing are
 *               those of posekf_replay_innovation_f32.  Then  NLL = (innov_acc[0] + innov_acc[1]) / 2 + 3/2 T ln 2 pi,
 *               mean NIS = innov_acc[0] / T (about 3 for a consistent model).
 *   innov_model POSEKF_INNOV_FULL or POSEKF_INNOV_TANGENT; any other value: POSEKF_EINVAL.
 * A buffer holds the sums of one model: pass it to launches of that model only. */
int posekf_replay_innovation_ex_f32(int64_t n_filters, int64_t n_steps, const float* streams, int64_t n_streams,
                                    const float* dt, int dt_per_step, const float* acc_ref, const float* mag_ref,
                                    const float* q_scale, const float* r_scale, float lpf_alpha_acc, float lpf_alpha_mag,
                                    float* state_x, float* state_x_lo, float* state_p, float* state_lpf, float* out_traj,
                                    uint8_t* out_flip, const float* truth, float* loss_acc, float* innov_acc, int innov_model,
                                    int wahba_algo, int staging, int state_flags, void* stream);

/* A batch of recordings in one launch, each with its own time steps and length (Python Kalman Filter/main_file.py:25,
 * 38-47: every recording differences its own timestamps against its own previousT).  The parameters of
 * posekf_replay_innovation_ex_f32, plus:
 *   dt_cols     [T][Ns] seconds, or NULL: filter n steps with dt_cols[t][n % Ns] (overrides dt / dt_per_step; dt may
 *               then be NULL).  Not 16-byte aligned: POSEKF_STAGE_AUTO runs the LDG kernel, an explicit TMA staging
 *               returns POSEKF_EALIGN (as for streams).
 *   n_valid     [Ns] int32, or NULL: stream c has n_valid[c] steps in this launch; the caller guarantees
 *               0 <= n_valid[c] <= T (it is not read on the host).  A step t >= n_valid[n % Ns] leaves filter n as it
 *               is: state, P, low-pass state, loss_acc and innov_acc are unchanged, the trajectory slot gets the held
 *               state (reference frame) and the flip byte is 0.  The samples and dt of such a step are never used:
 *               they may hold anything, NaN included.  For a time-chunked replay pass the lengths counted from the
 *               chunk's first step, clamped to [0, chunk length].
 *   innov_acc   may be NULL (no innovation sums); innov_model must be POSEKF_INNOV_FULL or POSEKF_INNOV_TANGENT.
 * With dt_cols and n_valid both NULL the call is posekf_replay_innovation_ex_f32 (innov_acc non-NULL) or
 * posekf_replay_f32 (innov_acc NULL).  Filters with all of their steps live give the same bits as one launch per
 * recording with that recording's dt[T]; every staging and variant is supported. */
int posekf_replay_batch_f32(int64_t n_filters, int64_t n_steps, const float* streams, int64_t n_streams, const float* dt,
                            int dt_per_step, const float* acc_ref, const float* mag_ref, const float* q_scale,
                            const float* r_scale, float lpf_alpha_acc, float lpf_alpha_mag, float* state_x, float* state_x_lo,
                            float* state_p, float* state_lpf, float* out_traj, uint8_t* out_flip, const float* truth,
                            float* loss_acc, float* innov_acc, int innov_model, int wahba_algo, int staging, int state_flags,
                            void* stream, const float* dt_cols, const int32_t* n_valid);

/* Innovation gating: the replay of posekf_replay_batch_f32 (same parameters, same rules) with outlier measurements
 * rejected by their tangent-space normalised innovation squared.  A live step is GATED iff
 *     NIS3_t = e3^T S3^-1 e3 > gate_nis3          (S = P^- + r I, e = y - z after the comparator, u = z/|z|; see
 *                                                  posekf_replay_innovation_ex_f32 for e3 and S3)
 * computed the same way whichever innov_model the launch accumulates.  The comparison is strict: a NaN statistic is
 * not gated (NaN propagates as in the reference).  Under a consistent model NIS3 ~ chi^2_3: 16.27 is its 0.999
 * quantile.  On a gated step:
 *   state       X_t = z_t / |z_t|, the normalised prediction (the update with e = 0); x_lo carries it the same way;
 *   covariance  P_t = P^-_t, the propagated covariance: state_p holds P^-/r;
 *   flip byte, loss_acc, low-pass state: as without the gate (the comparator still runs, the fix-up still applies);
 *   innov_acc   still adds the step's terms: the prediction-error decomposition stays the exact likelihood of the
 *               observations under the predictor that produced z and S, so the NLL stays a (Q,R) objective.
 * Held steps (t >= n_valid) are never gated and never counted.  gate_nis3 = +inf gives the bits of the same launch
 * without the gate; a chunked replay equals the unchunked one (the gate carries no state beyond X and P).  With q = 0
 * a run of rejected steps can never reopen the gate: P^- does not grow.
 *   gate_nis3   the threshold; NaN: POSEKF_EINVAL.
 *   gate_count  [N] int32 in/out, or NULL: += the number of gated steps of filter n (4-byte aligned, else
 *               POSEKF_EALIGN).
 *   out_gated   [T][N] uint8, or NULL: 1 where the step was gated, else 0 (held steps 0).
 * The packed kernel reads gate_count 8 bytes and writes out_gated 2 bytes at a time: buffers not aligned for that run
 * the scalar TMA kernel (same results).  Which kernel runs which combination: DESIGN.md section 5, f8. */
int posekf_replay_gated_f32(int64_t n_filters, int64_t n_steps, const float* streams, int64_t n_streams, const float* dt,
                            int dt_per_step, const float* acc_ref, const float* mag_ref, const float* q_scale,
                            const float* r_scale, float lpf_alpha_acc, float lpf_alpha_mag, float* state_x, float* state_x_lo,
                            float* state_p, float* state_lpf, float* out_traj, uint8_t* out_flip, const float* truth,
                            float* loss_acc, float* innov_acc, int innov_model, int wahba_algo, int staging, int state_flags,
                            void* stream, const float* dt_cols, const int32_t* n_valid, float gate_nis3, int32_t* gate_count,
                            uint8_t* out_gated);

/* Per-step innovation output: the replay of posekf_replay_gated_f32 (same parameters, same rules) that also writes the
 * terms each step adds to the innovation sums, so that a recording can be scored step by step or window by window
 * (where the filter is inconsistent, a gate threshold from a quantile of clean data, the likelihood of one segment).
 *   out_innov   [2][T][N] float32 (planes innov_plane_stride elements apart), required unless n_steps * n_filters = 0
 *               (NULL: POSEKF_EINVAL), 4-byte aligned (else POSEKF_EALIGN).  out_innov[0][t][n] = NIS_t, out_innov[innov_plane_stride + t N + n] =
 *               ln det S_t of filter n, in the convention of innov_acc: natural log, true units, without the
 *               (dof/2) ln 2 pi constant; the model is innov_model (POSEKF_INNOV_FULL: the 4-D terms,
 *               POSEKF_INNOV_TANGENT: NIS3_t and ln det S3_t).  Filter index fastest, like out_gated.
 *   innov_plane_stride  elements from plane 0 to plane 1, >= n_steps * n_filters (else POSEKF_EINVAL): a time chunk
 *               t0..t1 of a replay can write straight into its slice of a full-length [2][T_total][N] buffer (plane
 *               stride T_total N, base out_innov + t0 N).
 *   innov_acc   may be NULL: the launch then writes the per-step terms only.  With a buffer, both.
 * Held steps (t >= n_valid) write 0 to both planes, so for every filter sum_t out_innov[k][t][n] is what the launch adds
 * to innov_acc[k][n] up to float32 summation: ln det S_t is the addend of the sum itself, NIS_t the product the sum's
 * fused multiply-add adds, rounded on its own (one rounding per step apart).  Gated steps write their terms like any
 * other step; with POSEKF_INNOV_TANGENT plane 0 is the statistic the gate thresholded (the gate compares r NIS3 with
 * gate_nis3 r, so its decisions agree with out_innov[0] > gate_nis3 except at ties within rounding).
 * gate_nis3 = +inf with gate_count and out_gated NULL is an ungated launch.  Every other output (state, P, trajectory,
 * flips, loss, innov_acc, gate_count, out_gated) is bit-identical to the same launch without out_innov, and a chunked
 * replay writes what the unchunked one writes.  All three Wahba modes, both variants, the low-pass, per-stream dt and
 * lengths and the gate are supported; the scalar kernels run it (a packed staging runs the scalar TMA kernel, same bits).
 * With general Q and R matrices: posekf_replay_general_innovation_f32. */
int posekf_replay_innovation_steps_f32(int64_t n_filters, int64_t n_steps, const float* streams, int64_t n_streams,
                                       const float* dt, int dt_per_step, const float* acc_ref, const float* mag_ref,
                                       const float* q_scale, const float* r_scale, float lpf_alpha_acc, float lpf_alpha_mag,
                                       float* state_x, float* state_x_lo, float* state_p, float* state_lpf, float* out_traj,
                                       uint8_t* out_flip, const float* truth, float* loss_acc, float* innov_acc,
                                       int innov_model, int wahba_algo, int staging, int state_flags, void* stream,
                                       const float* dt_cols, const int32_t* n_valid, float gate_nis3, int32_t* gate_count,
                                       uint8_t* out_gated, float* out_innov, int64_t innov_plane_stride);

/* General Q and R matrices: the replay of posekf_replay_batch_f32 (same parameters and rules, minus q_scale / r_scale)
 * for filters whose process noise Q is any symmetric positive semidefinite 3x3 and whose measurement noise R is any
 * symmetric positive definite 4x4 -- the reference's KalmanFilter with its Q and R attributes assigned
 * (PKF/ExtendedKalmanFilter.py:58-80).  Each step is
 *     P^- = A P A^T + B(x) Q B(x)^T      (A = 0.5 Omega(w), the reference's own; B at the state before the step)
 *     z   = RK4 prediction               (restructured as in posekf_replay_f32, DESIGN.md section 3)
 *     S = P^- + R,  K = P^- S^-1,  y = the Wahba quaternion sign-fixed against z by the comparator
 *     X = (z + K (y - z)) / |.|,  P = P^- - K P^-.
 *   q_tri   [6][nq]: the upper triangle of Q, row-major (Q00 Q01 Q02 Q11 Q12 Q22); nq = 1 (one Q for the launch) or
 *           n_filters (filter n uses column n).  4-byte aligned, else POSEKF_EALIGN.
 *   r_tri   [10][nr]: the upper triangle of R in the order of state_p (R00 R01 R02 R03 R11 R12 R13 R22 R23 R33); nr = 1
 *           or n_filters.
 *   state_p holds P itself, NOT P/r as in the scalar entry points: convert when a state moves between the two.
 * Precondition (not checked here, like r > 0 and q >= 0 of the scalar entry points): R positive definite, Q positive
 * semidefinite, both symmetric.  POSEKF_EINVAL: innov_acc or state_x_lo non-NULL (no precise variant with general
 * matrices; the innovation sums, their per-step terms and the gate are posekf_replay_general_innovation_f32's), nq or
 * nr neither 1 nor n_filters, q_tri or r_tri NULL, and everything posekf_replay_batch_f32 refuses.  The float64 flip fix-up, the tuning loss (truth/loss_acc),
 * the low-pass, all three Wahba modes, per-stream dt / lengths and the filter-frame state flags work as in
 * posekf_replay_batch_f32.  A chunked replay equals the unchunked one bit for bit; every staging gives the same bits
 * (a packed staging runs the scalar TMA kernel).  The float32 step meets the 1e-5 rad tolerance of the float64
 * reference for eigenvalue ratios lambda(R)/lambda(Q) <= 100 and lambda(Q)/lambda(R) <= 1e4 (DESIGN.md, f9). */
int posekf_replay_general_f32(int64_t n_filters, int64_t n_steps, const float* streams, int64_t n_streams, const float* dt,
                              int dt_per_step, const float* acc_ref, const float* mag_ref, const float* q_tri, int64_t nq,
                              const float* r_tri, int64_t nr, float lpf_alpha_acc, float lpf_alpha_mag, float* state_x,
                              float* state_x_lo, float* state_p, float* state_lpf, float* out_traj, uint8_t* out_flip,
                              const float* truth, float* loss_acc, float* innov_acc, int innov_model, int wahba_algo,
                              int staging, int state_flags, void* stream, const float* dt_cols, const int32_t* n_valid);

/* General Q and R matrices with the innovation likelihood, its per-step terms and the innovation gate: the replay of
 * posekf_replay_general_f32 (same parameters, same rules for q_tri / nq / r_tri / nr, state_p holds P itself) plus the
 * tail of posekf_replay_innovation_steps_f32.  The filter steps exactly as posekf_replay_general_f32; on that step:
 *   4-D terms (innov_model POSEKF_INNOV_FULL)     NIS_t = e^T S^-1 e,  ln det S_t,   S = P^- + R,  e = sg y/|y| - z;
 *   tangent terms (POSEKF_INNOV_TANGENT)          NIS3_t = e3^T S3^-1 e3,  ln det S3_t,  e3 = E^T e,  S3 = E^T S E, E any
 *                                                 orthonormal basis of z-perp.
 * True units (natural log, without the (dof/2) ln 2 pi constant), as in every innovation entry point.
 *   innov_acc   [2][N] in/out or NULL: += sum_t NIS_t, sum_t ln det S_t.  Each sum adds exactly the float32 terms written
 *               to out_innov (one addition per step).
 *   out_innov, innov_plane_stride   as in posekf_replay_innovation_steps_f32, but out_innov may be NULL (no per-step
 *               output); with a buffer the stride must be >= n_steps * n_filters (else POSEKF_EINVAL), 4-byte alignment
 *               (else POSEKF_EALIGN).  Held steps write 0.
 *   gate_nis3, gate_count, out_gated   the gate of posekf_replay_gated_f32 on the tangent-space NIS3 in true units: a live
 *               step is gated iff NIS3_t > gate_nis3 (strict, NaN is never gated), and then keeps X_t = z_t/|z_t| and
 *               P_t = P^-_t; the flip byte, the loss, the low-pass, the sums and the per-step terms still see it.  With
 *               POSEKF_INNOV_TANGENT the decisions are exactly out_innov[0][t][n] > gate_nis3.  NaN gate_nis3:
 *               POSEKF_EINVAL.  +inf with gate_count and out_gated NULL is an ungated launch.
 * Every other output is bit-identical to posekf_replay_general_f32 on the same inputs when the launch is ungated, and a
 * chunked replay equals the unchunked one bit for bit (sums, counts, per-step slices).  Any combination of innov_acc,
 * out_innov and the gate may be asked for; with none of them the launch is posekf_replay_general_f32's.  All three Wahba
 * modes, the low-pass, per-stream dt / lengths and the state flags work as there; every staging gives the same bits (a
 * packed staging runs the scalar TMA kernel).  POSEKF_EINVAL also for state_x_lo non-NULL (no precise variant with
 * general matrices) and an unknown innov_model. */
int posekf_replay_general_innovation_f32(int64_t n_filters, int64_t n_steps, const float* streams, int64_t n_streams,
                                         const float* dt, int dt_per_step, const float* acc_ref, const float* mag_ref,
                                         const float* q_tri, int64_t nq, const float* r_tri, int64_t nr, float lpf_alpha_acc,
                                         float lpf_alpha_mag, float* state_x, float* state_x_lo, float* state_p,
                                         float* state_lpf, float* out_traj, uint8_t* out_flip, const float* truth,
                                         float* loss_acc, float* innov_acc, int innov_model, int wahba_algo, int staging,
                                         int state_flags, void* stream, const float* dt_cols, const int32_t* n_valid,
                                         float gate_nis3, int32_t* gate_count, uint8_t* out_gated, float* out_innov,
                                         int64_t innov_plane_stride);

/* Same replay with HOST buffers: streams_host [T][9][N] is streamed through the device in time
 * chunks (double-buffered H2D copies overlapped with the filter kernel, state carried across
 * chunks on the device), results are copied back.  This is the call an offline-replay user makes.
 *   out_x_host [4][N], out_p_host [10][N] = upper triangle of P itself, unscaled (may be NULL), out_traj_host [T][N][4] (may be NULL).
 *   x0_host / p0_host ([4][N] / [10][N] upper triangle of P, unscaled) may be NULL (X=[1,0,0,0], P=I4:
 *   PKF/main_file.py:23,26).
 *   precise     non-zero selects the precise variant (see state_x_lo of posekf_replay_f32) for extreme Q/R.
 *   chunk_steps  steps per chunk when no workspace is given (0 = about 256 MiB per staging buffer).
 *   device      CUDA device ordinal.
 *   workspace   from posekf_host_workspace_create (staging buffers, streams and events are reused across
 *               calls -- allocating and freeing GiB-sized buffers per call costs tens of ms), or NULL
 *               for a temporary one.
 * Host buffers should be page-locked (cudaHostAlloc / cudaHostRegister) for full PCIe rate.
 * Every r_scale must be > 0 and every q_scale >= 0 (checked on the host: POSEKF_EINVAL otherwise).  The caller's current
 * CUDA device is restored before returning; on a failure all work issued so far is drained before the call returns. */
int posekf_replay_host_f32(int64_t n_filters, int64_t n_steps, const float* streams_host, float dt,
                           const float* acc_ref_host, const float* mag_ref_host, const float* q_scale_host,
                           const float* r_scale_host, float lpf_alpha_acc, float lpf_alpha_mag,
                           const float* x0_host, const float* p0_host, float* out_x_host, float* out_p_host,
                           float* out_traj_host, int64_t chunk_steps, int wahba_algo, int precise, int device,
                           void* workspace);

/* Reusable workspace of posekf_replay_host_f32 for batches of n_filters on `device` (the only objects
 * this library ever allocates).  chunk_steps <= 0 picks ~256 MiB staging buffers. */
int posekf_host_workspace_create(int device, int64_t n_filters, int64_t chunk_steps, int with_trajectory, void** out_ws);
int posekf_host_workspace_destroy(void* workspace);

/* ---------------------------------------------------------------------------------------------
 * Wahba.getRotation / Wahba.getQuarternion for N (acc, mag) pairs.   PKF/Wahba.py:8-17,49-50
 *   acc_ref, mag_ref  [3][N], or [3] when ref_shared != 0 (one Wahba object, PKF/Wahba.py:4-6)
 *   acc, mag    [3][N]
 *   k_acc,k_mag [N] weights, or NULL: then the scalars k_acc_s / k_mag_s are used, or, when
 *               weights_from_acc != 0, the reference's k_acc=|acc_z|, k_mag=1-|acc_z|
 *               (PKF/ExtendedKalmanFilter.py:71)
 *   out_rot     [9][N] rotation matrix (row-major) or NULL;  out_quat [4][N] or NULL
 *   jacobi_sweeps  accepted for interface compatibility and ignored: the QR-preconditioned Jacobi SVD works on a
 *               2x2 core, for which ONE rotation is exact
 */
int posekf_wahba_f32(int64_t n, const float* acc_ref, const float* mag_ref, int ref_shared, const float* acc,
                     const float* mag, const float* k_acc, const float* k_mag, float k_acc_s, float k_mag_s,
                     int weights_from_acc, float* out_rot, float* out_quat, int wahba_algo, int jacobi_sweeps,
                     void* stream);

/* Comparison tracks of the tuning workflow (the curves the reference plots beside the filter,
 * PKF/main_file.py:40-46,50-52 and the Results/ plots): for N filters over T steps of the same stream
 * layout as posekf_replay_f32,
 *   out_gyro  [T][N][4]  gyro-only attitude: RK4 without correction from gyro_state (X=[1,0,0,0] when
 *             gyro_state is NULL)   -- SRV/KalmanFilter.cpp:149 `Quarternion_Gyro_pure`
 *   out_wahba [T][N][4]  Wahba-only attitude per sample, reference sign convention
 *             -- PKF/main_file.py:40 getQuarternion(acc, mag, k_acc=.5, k_mag=.5); weights_from_acc != 0
 *             selects the filter's own |acc_z|, 1-|acc_z| instead
 *   gyro_state [4][N] in/out (carried across time chunks) or NULL.   Either output may be NULL. */
int posekf_tracks_f32(int64_t n_filters, int64_t n_steps, const float* streams, int64_t n_streams, const float* dt,
                      int dt_per_step, const float* acc_ref, const float* mag_ref, float k_acc, float k_mag,
                      int weights_from_acc, float* gyro_state, float* out_gyro, float* out_wahba, int wahba_algo,
                      void* stream);

/* Raw-sensor pre-processing in front of the filter (online pipeline, SRV/Parser.cpp:229-267):
 * per filter and gyro sample, linearly interpolate the accel / mag samples that bracket the gyro
 * timestamp  y = (y2 - y1)/(t2 - t1)*(t3 - t1) + y1  (LinearInterpolationSensor, :259-267), normalise
 * (NormalizeValues, :221-228), optionally low-pass with alpha (SRV/KalmanFilter.cpp:279-303; < 0 = off;
 * then leave lpf off in posekf_replay_f32) and write the [T][9][N] stream of posekf_replay_f32.
 *   gyro [T][3][N]; raw_prev, raw_next [T][6][N] (acc xyz, mag xyz before / after the gyro timestamp);
 *   tspan [T][4][N] seconds: acc (t2-t1), acc (t3-t1), mag (t2-t1), mag (t3-t1) -- differenced from the
 *   integer ns timestamps by the caller; lpf_state [6][N] in/out (start at 0) or NULL. */
int posekf_preprocess_f32(int64_t n_filters, int64_t n_steps, const float* gyro, const float* raw_prev,
                          const float* raw_next, const float* tspan, float lpf_alpha_acc, float lpf_alpha_mag,
                          float* lpf_state, float* out_streams, void* stream);

/* Initial reference vectors of the online pipeline: mean and (optionally) unbiased variance of the first K
 * samples of a sensor for N recordings; normalize != 0 divides the mean by its norm, which is how acc_0 / mag_0
 * are produced (SRV/InitialValues.cpp:19-66, SRV/Parser.cpp:46-49; K = 100 there, SRV/Parser.cpp:5-7).
 *   samples [K][3][N] -> out_mean [3][N], out_var [3][N] or NULL (variance of the raw samples, K >= 2). */
int posekf_initial_values_f32(int64_t n_filters, int64_t n_samples, const float* samples, int normalize, float* out_mean,
                              float* out_var, void* stream);

/* Raw event recordings -> the batch of posekf_replay_batch_f32 (what SRV/Parser.cpp:148-267 does per event, for a
 * batch of recordings in one call; DESIGN section 5 f10).
 * Input: n_rec recordings, each with a gyro, an accelerometer and a magnetometer event stream.  Per sensor s the
 * streams are concatenated: t_s [M_s] int64 ns, v_s [3][M_s] float32, off_s [n_rec+1] int64; recording c owns events
 * off_s[c] .. off_s[c+1]-1 and M_s = off_s[n_rec].  PRECONDITION (not checked here, like n_valid of
 * posekf_replay_batch_f32): timestamps strictly increase within each recording's stream, and each recording has fewer
 * than 2^31 gyro events.
 *   acc_ref / mag_ref [3][n_rec]: the normalised means of the recording's first k_init acc / mag events (float64 sums in
 *     arrival order, as posekf_initial_values_f32; k_init = 100 in SRV/Parser.cpp:5-7).  t_init: the later of the two
 *     k_init-th timestamps.  A recording with fewer than k_init events of either sensor has length 0 and the
 *     references (0,0,1) / (1,0,0).
 *   lengths [n_rec] int32: the number of steps.  The steps are the gyro events g with t_g > t_init that both sensors
 *     bracket (an event at t1 <= t_g and one at t2 > t_g); they are consecutive gyro events.
 *   streams [t_out][9][n_rec]: step i of recording c is gyro event i of its steps, with acc and mag interpolated from
 *     the LAST event at or before t_g and the FIRST event after it and normalised, with the operations of
 *     posekf_preprocess_f32 (same device function); t2 - t1 and t_g - t1 are differenced in int64 ns, then converted
 *     to float seconds as (float)(d * 1e-9) in double.
 *   dt_cols [t_out][n_rec] seconds: (t_g(i) - t_g(i-1)) * 1e-9, and (t_g(0) - t_init) * 1e-9 for step 0, differenced
 *     in int64 and rounded to float32 once.
 *   Steps i >= lengths[c] (padding, never read by a replay with n_valid = lengths): the last step repeated with dt 0;
 *     for a recording of length 0, gyro 0 and its reference vectors (the convention of logio.stack_logs).
 * Query mode: streams NULL writes lengths only (the values, dt_cols and the references may be NULL), so that the caller
 * can size t_out >= max(lengths) with one read-back.  With t_out < max(lengths) only the first t_out steps are written.
 * POSEKF_EINVAL: n_rec < 0, t_out < 0, k_init < 1, or a NULL required pointer. */
int posekf_align_events_f32(int64_t n_rec, int64_t k_init, const int64_t* gyro_t, const float* gyro_v, const int64_t* gyro_off,
                            const int64_t* acc_t, const float* acc_v, const int64_t* acc_off, const int64_t* mag_t,
                            const float* mag_v, const int64_t* mag_off, int64_t t_out, float* streams, float* dt_cols,
                            int32_t* lengths, float* acc_ref, float* mag_ref, void* stream);

/* Measurement stream for POSEKF_WAHBA_PRECOMPUTED.  The Wahba solution of a sample does not depend on Q or R,
 * so a tuning sweep that replays Ns trajectories N/Ns times solves it ONCE per (trajectory, step):
 *   streams [T][9][Ns] (gyro, acc, mag) -> out_streams [T][9][Ns]: rows 0-2 gyro, rows 3-6 the quaternion of
 *   Wahba.getQuarternion(acc, mag, |acc_z|, 1-|acc_z|) in the reference's sign convention
 *   (PKF/ExtendedKalmanFilter.py:71, PKF/Wahba.py:49-50), rows 7-8 zero.
 * The optional low-pass (alpha >= 0, lpf_state [6][Ns] in/out) is applied here, before the solve; the replay of
 * a measurement stream must then run with the low-pass off.  wahba_algo: POSEKF_WAHBA_QR2 or _JACOBI. */
int posekf_measurement_stream_f32(int64_t n_streams, int64_t n_steps, const float* streams, const float* acc_ref,
                                  const float* mag_ref, float lpf_alpha_acc, float lpf_alpha_mag, float* lpf_state,
                                  float* out_streams, int wahba_algo, void* stream);

/* Quart2RPY over a stored trajectory: traj [M][4] (e.g. out_traj with M = T*N) -> degrees [M][3].
 * PKF/UtilityFunctions.py:3-14; C++ twin SRV/KalmanFilter.cpp:194-233 (which clamps asin; this does not,
 * like the Python oracle). */
int posekf_traj2rpy_f32(int64_t m, const float* traj, float* out_rpy_deg, void* stream);

/* Wahba.RotationMatrix2Quart for N matrices: rot [9][N] -> quat [4][N].   PKF/Wahba.py:20-47 */
int posekf_rot2quat_f32(int64_t n, const float* rot, float* out_quat, void* stream);

/* ---------------------------------------------------------------------------------------------
 * KalmanFilter.Prediction for N filters, general matrices.   PKF/ExtendedKalmanFilter.py:58-68
 *   gyro [3][N]; dt [N] seconds (dt_shared=0) or one float (dt_shared=1); x [4][N]; p [16][N];
 *   q_mat [9], r_mat [16] shared by all filters; q_scale/r_scale [N] optional per-filter multipliers
 *   (NULL = 1) so that Q_n = q_scale[n]*q_mat.   Outputs z [4][N], p_out [16][N], k_out [16][N].
 */
int posekf_predict_f32(int64_t n, const float* gyro, const float* dt, int dt_shared, const float* x, const float* p,
                       const float* q_mat, const float* r_mat, const float* q_scale, const float* r_scale,
                       float* out_z, float* out_p, float* out_k, void* stream);

/* KalmanFilter.Correction for N filters, general P and K.   PKF/ExtendedKalmanFilter.py:70-80
 *   mag, acc [3][N] (NB the reference's argument order is Mag, Acc); acc_ref/mag_ref as in
 *   posekf_wahba_f32; z [4][N]; p,k [16][N].  Outputs x [4][N], p_out [16][N], out_flip [N] uint8 or
 *   NULL, out_meas [4][N] (the sign-fixed Wahba quaternion) or NULL.
 */
int posekf_correct_f32(int64_t n, const float* mag, const float* acc, const float* acc_ref, const float* mag_ref,
                       int ref_shared, const float* z, const float* p, const float* k, float* out_x, float* out_p,
                       uint8_t* out_flip, float* out_meas, int wahba_algo, void* stream);

/* KalmanFilter.RungeKutta4 (static) for N states: q [4][N], dt seconds, w [3][N] -> out_q [4][N].
 * PKF/ExtendedKalmanFilter.py:25-41 (the reference's T is in ns and is scaled by 1e-9 at :32). */
int posekf_rk4_f32(int64_t n, const float* q, const float* dt, int dt_shared, const float* w, float* out_q,
                   void* stream);

/* GetJacobian_A / GetJacobian_B: w [3][N] -> a [16][N];  q [4][N] -> b [12][N] (4x3 row-major).
 * PKF/ExtendedKalmanFilter.py:43-48, :51-56.  Either pair may be NULL. */
int posekf_jacobians_f32(int64_t n, const float* w, float* out_a, const float* q, float* out_b, void* stream);

/* KalmanFilter.Comparator: conj(q1) (x) q2 for N pairs, [4][N] each.  PKF/ExtendedKalmanFilter.py:16-23 */
int posekf_comparator_f32(int64_t n, const float* q1, const float* q2, float* out, void* stream);

/* Low-pass y <- alpha x + (1-alpha) y along time for N channels-triples.
 * x [T][3][N] -> out [T][3][N] (may alias x); state [3][N] in/out (start at 0 like
 * SRV/KalmanFilter.cpp:16-18 / PKF/Test.py:7-9).   SRV/KalmanFilter.cpp:21-24, PKF/Test.py:27-33 */
int posekf_lowpass_f32(int64_t n, int64_t n_steps, const float* x, float alpha, float* state, float* out,
                       void* stream);

/* UtilityFunctions.Quart2RPY for N quaternions: q [4][N] -> rpy degrees [3][N] (asin not clamped).
 * PKF/UtilityFunctions.py:3-14 */
int posekf_quat2rpy_f32(int64_t n, const float* q, float* out_rpy_deg, void* stream);

/* UtilityFunctions.norm for N vectors of length k: v [k][N] -> out [N].  PKF/UtilityFunctions.py:16-21 */
int posekf_norm_f32(int64_t n, int k, const float* v, float* out, void* stream);

/* Plumbing for hosts that bind this library without a CUDA runtime binding of their own (the
 * reference-named Python modules use them for their per-call staging): an asynchronous copy between a
 * (preferably page-locked) host buffer and device memory on `stream`, and a stream synchronise. */
int posekf_copy_async(void* dst, const void* src, int64_t bytes, int to_device, void* stream);
int posekf_stream_sync(void* stream);

/* Measurement helper (not in the reference): runs a register-resident FFMA loop on every SM and
 * returns the achieved FP32 rate in TFLOP/s (2 flop per FFMA) -- the denominator of the FP32
 * roofline, measured in the same process and at the same clocks as the filter kernel. */
int posekf_fp32_peak_tflops(int device, double* out_tflops, double* out_ms);

#ifdef __cplusplus
}
#endif
#endif /* POSEKF_H_ */
