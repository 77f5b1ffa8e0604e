/* rbm_b200.h -- C ABI of librbm_b200.so: batched rigid-body inverse dynamics on NVIDIA B200 (sm_100a).
 *
 * The reference (barikata1984/rigid-body-manipulation) has NO FFI layer: its hot path is a set of plain
 * Python module functions (dynamics/dynamics.py, transformations/transformations.py) working on numpy
 * arrays and liegroups objects.  This header is therefore the boundary a maintainer would bind from
 * Python with ctypes (INTEGRATION.md shows the stub); each entry point names the reference function
 * (file:line) it replaces.  Conventions:
 *
 *   - plain pointers and sizes only; no C++ / torch types
 *   - model constants are HOST pointers (tiny, copied once); batch buffers are DEVICE pointers unless the
 *     function name ends in _host
 *   - twists / wrenches are 6-vectors in [linear(3); angular(3)] order, as in the reference (liegroups order)
 *   - poses are 12 scalars: rotation row-major (9) then translation (3)
 *   - SoA batch layout: element (j, s) of a [k][ld] array is at base[j*ld + s], s = sample index < n <= ld
 *   - AoS batch layout mirrors the reference's `traj` argument: traj[s][3][nj] = (q, qd, qdd) rows
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*; NULL = default stream);
 *     return value 0 = ok, negative = rbm_status; the message is in rbm_last_error_string()
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails with RBM_ERR_CUDA
 */
#ifndef RBM_B200_H
#define RBM_B200_H

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define RBM_API __attribute__((visibility("default")))
#else
#define RBM_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef struct rbm_model rbm_model; /* opaque: model constants resident on one device */

typedef enum rbm_status {
  RBM_OK = 0,
  RBM_ERR_INVALID = -1,     /* bad argument (maps to AssertionError / ValueError in the Python shim) */
  RBM_ERR_CUDA = -2,        /* CUDA runtime error, incl. "no device" */
  RBM_ERR_UNSUPPORTED = -3, /* e.g. nj > RBM_MAX_JOINTS */
  RBM_ERR_NCCL = -4
} rbm_status;

enum { RBM_MAX_JOINTS_ABI = 16 };

/* rbm_model_create flags */
enum {
  RBM_FLAG_FORCE_GENERIC = 1, /* never select a structure-specialised kernel */
  RBM_FLAG_NO_TMA = 2         /* never use the bulk-async (TMA) pipelined kernel variants */
};

/* kernel path chosen for a model (rbm_model_kernel_path) */
enum {
  RBM_PATH_GENERIC = 0,   /* any chain: dense inertias, arbitrary screws / poses (shared-memory parameters) */
  RBM_PATH_SEQ_ISO = 1,   /* the reference's sequential.xml structure, links 1-5 isotropic, link 6 rigid body */
  RBM_PATH_SEQ_RIGID = 2  /* same kinematic structure, every link a general rigid body */
};

RBM_API const char* rbm_version(void);
RBM_API const char* rbm_last_error_string(void); /* thread-local */
RBM_API int rbm_device_count(void);              /* 0 when no CUDA device / driver is present */
/* PCI bus id ("0000:1b:00.0"-style, lower-cased by the caller for sysfs) of a CUDA device, as the runtime numbers it (i.e. after
 * CUDA_VISIBLE_DEVICES).  Host plumbing for NUMA placement of the pinned buffers the *_host entry points stream from. */
RBM_API int rbm_device_pci_bus_id(int device, char* out, int len);

/* ---- model ------------------------------------------------------------------------------------------
 * Binds the arguments that reference core/simulate.py:150-156 binds with functools.partial onto
 * dynamics.inverse (dynamics/dynamics.py:109-118):
 *   hposes_Rt  [(nj+1)][12]  hposes_body_parent (entry 0 unused, dynamics.py:125)
 *   simats     [(nj+1)][36]  simats_body, row-major 6x6 (entry 0 unused, dynamics.py:144)
 *   uscrews    [nj][6]       uscrews_body
 *   twist_0, dtwist_0 [6]
 *   wrench_tip [6] or NULL (= zeros, dynamics.py:116);  pose_tip_Rt [12] or NULL (= identity, :117)
 *   pose_sen_Rt [12] or NULL (= identity): static pose of the F/T sensor frame w.r.t. the last link's joint
 *                frame, pose_sen_llj of core/simulate.py:202 (used by the regressor entry points only)
 * The constants are copied; the caller keeps ownership of its arrays.  `device` is the CUDA ordinal. */
RBM_API int rbm_model_create(int nj, const double* hposes_Rt, const double* simats, const double* uscrews, const double* twist_0,
                     const double* dtwist_0, const double* wrench_tip, const double* pose_tip_Rt, const double* pose_sen_Rt,
                     unsigned flags, int device, rbm_model** out);
RBM_API void rbm_model_destroy(rbm_model* m);
/* Device-free analysis of the same constants (needs no GPU): which kernel path the model takes and the parameter blocks the
 * kernels would receive -- fast_params [rbm_fast_param_count()] (the structure-specialised kernels' constant block, zeros when the
 * path is generic) and generic_params [rbm_generic_param_count(nj)] (the shared-memory block of the generic kernels).  Any output
 * pointer may be NULL.  Validation and error codes are those of rbm_model_create. */
RBM_API int rbm_model_analyze(int nj, const double* hposes_Rt, const double* simats, const double* uscrews, const double* twist_0,
                      const double* dtwist_0, const double* wrench_tip, const double* pose_tip_Rt, const double* pose_sen_Rt,
                      unsigned flags, int* kernel_path, double* fast_params, double* generic_params);
RBM_API int rbm_fast_param_count(void);
RBM_API int rbm_generic_param_count(int nj);
RBM_API int rbm_model_num_joints(const rbm_model* m);
RBM_API int rbm_model_kernel_path(const rbm_model* m);

/* ---- inverse dynamics -------------------------------------------------------------------------------
 * Batched dynamics.inverse (dynamics/dynamics.py:109-157): tau[j][s] for every sample s.
 *   q, qd, qdd : [nj][ld]   tau : [nj][ld]
 *   twist_last, dtwist_last : [6][ld] or NULL -- V and dV of the last link (twists[nj], dtwists[nj] of
 *   the reference's return value; the only entries core/simulate.py:203,206 reads).
 * On a fast-path model the kernels never read the gantry positions q[0..2], and a call without twists does not read the gantry
 * velocities qd[0..2] either (tau does not depend on them): the caller may leave those rows unset. */
RBM_API int rbm_rnea_f64(const rbm_model* m, const double* q, const double* qd, const double* qdd, double* tau, double* twist_last,
                 double* dtwist_last, int64_t n, int64_t ld, void* stream);
RBM_API int rbm_rnea_f32(const rbm_model* m, const float* q, const float* qd, const float* qdd, float* tau, float* twist_last,
                 float* dtwist_last, int64_t n, int64_t ld, void* stream);

/* Same, array-of-samples layout of the reference's own argument: traj [n][3][nj] -> tau [n][nj]. */
RBM_API int rbm_rnea_aos_f64(const rbm_model* m, const double* traj, double* tau, int64_t n, void* stream);
RBM_API int rbm_rnea_aos_f32(const rbm_model* m, const float* traj, float* tau, int64_t n, void* stream);

/* Full return value of dynamics.inverse (dynamics.py:157) per sample, AoS:
 *   traj [n][3][nj] -> tau [n][nj], poses [n][nj][12] (T_{i,i-1}, dynamics.py:126; the appended tip pose is the
 *   model's constant), twists [n][nj+1][6], dtwists [n][nj+1][6] (entry 0 = twist_0 / dtwist_0).
 *   Any of poses / twists+dtwists may be NULL (twists and dtwists only together). */
RBM_API int rbm_rnea_full_f64(const rbm_model* m, const double* traj, double* tau, double* poses, double* twists, double* dtwists,
                      int64_t n, void* stream);

/* The same with HOST buffers, for small batches (the scalar drop-in `dynamics.inverse` calls it with n = 1): one host->device
 * copy, one launch, one device->host copy through scratch owned by the model; synchronous.  poses / twists+dtwists may be NULL. */
RBM_API int rbm_rnea_full_host_f64(const rbm_model* m, const double* traj_host, double* tau_host, double* poses_host, double* twists_host,
                           double* dtwists_host, int64_t n);

/* Planner-driven inverse dynamics: the quintic rest-to-rest trajectory of planners/joint_position_planner.py:86-131
 * (traj_5th_spline) is evaluated inside the kernel, so nothing is read from HBM.  Sample s is step k = step0 + s*stride:
 *   prof = coeffs . [k^5 .. 1];  q_j = disp_j prof + offset_j;  qd_j = disp_j prof' / timestep;  qdd_j = disp_j prof'' / timestep^2
 * coeffs [6], disp [nj], offset [nj] are HOST pointers (the six coefficients come from the planner's own 6x6 solve).
 *   tau : [nj][ld];   traj : [3*nj][ld] (rows q_0..q_nj-1, qd_*, qdd_*) or NULL. */
RBM_API int rbm_rnea_planned_f64(const rbm_model* m, const double* coeffs, const double* disp, const double* offset, double timestep, double step0,
                         double stride, double* tau, double* traj, int64_t n, int64_t ld, void* stream);
RBM_API int rbm_rnea_planned_f32(const rbm_model* m, const double* coeffs, const double* disp, const double* offset, double timestep, double step0,
                         double stride, float* tau, float* traj, int64_t n, int64_t ld, void* stream);

/* End-to-end convenience for host callers (the `e2e` measurement): traj_host [n][3][nj] and tau_host [n][nj] are HOST
 * buffers (pinned memory gives full PCIe rate); copies host->device, runs the AoS kernel and copies back in
 * `chunk`-sample pieces on internal streams so transfers overlap compute.  Synchronous: returns when tau_host is
 * complete.  chunk <= 0 picks a default. */
RBM_API int rbm_rnea_host_f64(const rbm_model* m, const double* traj_host, double* tau_host, int64_t n, int64_t chunk);
RBM_API int rbm_rnea_host_f32(const rbm_model* m, const float* traj_host, float* tau_host, int64_t n, int64_t chunk);

/* Which rows of (q, qd, qdd) the model's inverse-dynamics kernels read when every output (tau, V_6, dV_6) is asked for: mask [3][nj],
 * 1 = live, 0 = the result does not depend on it and the kernel never loads it.  For the reference's structure (three leading
 * prismatic joints, core/simulate.py:98-110, xml_models/manipulators/sequential.xml:13-39) tau, V_6 and dV_6 do not depend on the
 * gantry positions q_0..q_2, so 15 of the 18 input rows are live.  A tau-only call reads three rows fewer: tau does not depend on
 * the gantry velocities qd_0..qd_2 either (a Galilean boost, no rotation precedes those joints), so it loads 12 rows -- 144
 * instead of 192 bytes of DRAM traffic per fp64 sample -- and rbm_rnea_host_soa_* uploads those 12. */
RBM_API int rbm_model_live_inputs(const rbm_model* m, int32_t* mask);

/* The same end-to-end path for the kernels' own SoA layout (what dynamics.inverse would be handed by a caller that batches a
 * whole trajectory: rows of q, qd, qdd): q_host, qd_host, qdd_host, tau_host are HOST buffers [nj][ld].  Only the rows the tau-only
 * kernel reads are uploaded (on a fast-path model: not q[0..2], not qd[0..2], which the caller may leave unset; see
 * rbm_model_live_inputs) -- one strided cudaMemcpy2DAsync per run of live rows and chunk -- and tau comes back
 * with one strided copy per chunk, both overlapped with the kernel over three internal streams.  Synchronous. */
RBM_API int rbm_rnea_host_soa_f64(const rbm_model* m, const double* q_host, const double* qd_host, const double* qdd_host, double* tau_host,
                          int64_t n, int64_t ld, int64_t chunk);
RBM_API int rbm_rnea_host_soa_f32(const rbm_model* m, const float* q_host, const float* qd_host, const float* qdd_host, float* tau_host, int64_t n,
                          int64_t ld, int64_t chunk);

/* Planner-driven end to end (planners/joint_position_planner.py:86-131 feeding dynamics.inverse, core/simulate.py:187-188): the
 * trajectory is generated inside the kernel as in rbm_rnea_planned_*, so nothing is uploaded; tau_host [nj][ld] is a HOST buffer
 * filled chunk by chunk while the next chunk computes.  Synchronous. */
RBM_API int rbm_rnea_planned_host_f64(const rbm_model* m, const double* coeffs, const double* disp, const double* offset, double timestep,
                              double step0, double stride, double* tau_host, int64_t n, int64_t ld, int64_t chunk);
RBM_API int rbm_rnea_planned_host_f32(const rbm_model* m, const double* coeffs, const double* disp, const double* offset, double timestep,
                              double step0, double stride, float* tau_host, int64_t n, int64_t ld, int64_t chunk);

/* ---- sensor-frame regressor and identification ------------------------------------------------------
 * Parameter order phi = [m, m cx, m cy, m cz, Ixx, Iyy, Izz, Ixy, Iyz, Izx] (dynamics.py:225-230, loggers.py:133),
 * inertia about the sensor-frame origin; regressor rows are [force (3); torque (3)]. */

/* get_regressor_matrix (dynamics/dynamics.py:215-249), batched, AoS: twists, dtwists [n][6] -> Y [n][6][10]. */
RBM_API int rbm_regressor_rows_f64(const double* twists, const double* dtwists, double* Y, int64_t n, void* stream);

/* Twists of the last link into the sensor frame (core/simulate.py:202-209), AoS [n][6]:
 * V_s = Ad(T) V, dV_s = Ad(T) dV with T = pose_Rt (HOST pointer, 12 scalars). */
RBM_API int rbm_sensor_twists_f64(const double* pose_Rt, const double* twists, const double* dtwists, double* twists_sen, double* dtwists_sen,
                          int64_t n, void* stream);

/* Fused (q, qd, qdd) [nj][ld] -> forward sweep -> sensor frame (the model's pose_sen_Rt) -> any of:
 *   Y          [n][6][10]  materialised regressor rows               (NULL to skip)
 *   twist_sen, dtwist_sen [6][ld]                                     (NULL to skip, only together)
 *   wrench     [6][ld] = Y phi with phi a DEVICE pointer to 10 scalars (both NULL to skip): the load a body with
 *              parameters phi puts on the sensor -- used to synthesise F/T data for identification benchmarks. */
RBM_API int rbm_regressor_from_traj_f64(const rbm_model* m, const double* q, const double* qd, const double* qdd, double* Y, double* twist_sen,
                                double* dtwist_sen, const double* phi, double* wrench, int64_t n, int64_t ld, void* stream);
RBM_API int rbm_regressor_from_traj_f32(const rbm_model* m, const float* q, const float* qd, const float* qdd, float* Y, float* twist_sen,
                                float* dtwist_sen, const float* phi, float* wrench, int64_t n, int64_t ld, void* stream);

/* Normal equations of the stacked least-squares problem of loggers/loggers.py:127-129 without materialising Y:
 *   gram_pack [112] (device, always double) = [Y^T Y (100, row-major) | Y^T f (10) | f^T f | n]
 *   f [6][ld]: measured wrench per sample in the sensor frame.
 *   workspace: device scratch of rbm_gram_workspace_bytes() bytes (per-block partial sums; no atomics, the
 *   reduction order is fixed, so results are bit-reproducible for a given n).
 * The fp32 entry point reads float inputs, forms the regressor in float and accumulates in double every 64 samples. */
RBM_API size_t rbm_gram_workspace_bytes(const rbm_model* m, int64_t n);
RBM_API int rbm_regressor_gram_f64(const rbm_model* m, const double* q, const double* qd, const double* qdd, const double* f, double* gram_pack,
                           void* workspace, size_t workspace_bytes, int64_t n, int64_t ld, void* stream);
RBM_API int rbm_regressor_gram_f32(const rbm_model* m, const float* q, const float* qd, const float* qdd, const float* f, double* gram_pack,
                           void* workspace, size_t workspace_bytes, int64_t n, int64_t ld, void* stream);

/* One Gram pack per GROUP (environment / object) for logs stored frame-major: sample `fr` of group g has its row k at
 *   x[fr * frame_stride + k * ld + g]  (x = q, qd, qdd: nj rows)   and   f[fr * f_frame_stride + k * ld + g]  (6 rows)
 * e.g. the frame log of rbm_closed_loop_f64 (q = frames, qd = frames + nj ld, qdd = frames + 2 nj ld, f = frames + (3 nj + 12) ld,
 * frame_stride = f_frame_stride = (3 nj + 18) ld), or the same trajectories with a separately stored (noisy) wrench array.  One group per thread, no workspace;  gram_packs: [112][ld_out], column g = the pack of group g. */
RBM_API int rbm_regressor_gram_grouped_f64(const rbm_model* m, const double* q, const double* qd, const double* qdd, const double* f, int64_t frame_stride,
                                   int64_t f_frame_stride, int64_t n_frames, double* gram_packs, int64_t n_groups, int64_t ld, int64_t ld_out, void* stream);

/* ---- the one collective: all-reduce of the Gram pack over NCCL ------------------------------------------------
 * Each rank accumulates the pack of its shard (rbm_regressor_gram_*), then rbm_allreduce_gram sums the 112 doubles in place
 * across ranks on `stream` (enqueue it right behind the Gram call: no host synchronisation is needed in between).
 * NCCL is resolved with dlopen at first use (libnccl.so.2); rbm_nccl_available() == 0 when it cannot be found.
 * Communicator set-up: rank 0 calls rbm_nccl_unique_id (128 bytes), the application broadcasts those bytes, every rank calls
 * rbm_nccl_comm_create (collective).  `comm` is an opaque ncclComm_t. */
RBM_API int rbm_nccl_available(void);
RBM_API int rbm_nccl_unique_id(void* id128);
RBM_API int rbm_nccl_comm_create(const void* id128, int nranks, int rank, int device, void** comm);
RBM_API int rbm_nccl_comm_destroy(void* comm);
RBM_API int rbm_allreduce_gram(void* comm, double* gram_pack, void* stream);
/* grouped form: `count` consecutive packs (one per object), one collective */
RBM_API int rbm_allreduce_gram_n(void* comm, double* gram_packs, int64_t count, void* stream);

/* ---- LQR linearisation ------------------------------------------------------------------------------------
 * Replaces dynamics.StateSpace.update_matrices (dynamics/dynamics.py:41-46 -> mjd_transitionFD, consumed by
 * controllers/lqr.py:43-49) for the reference's plant (nv = nu = nj, unit-gear motors, semi-implicit Euler with
 * step dt): x = [q; qd], x+ = f(x, u);  A = df/dx (2nj x 2nj), B = df/du (2nj x nj), by finite differences of the
 * batched inverse dynamics (step eps, centred or forward -- StateSpaceConfig.epsilon / .centered, dynamics.py:14-17).
 *   q, qd : [nj][ld];  u : [nj][ld] applied joint forces (ctrl), or NULL = zeros
 *   A : [(2nj*2nj)][ld] element-major: entry (r, c) of state s at A[(r*2nj + c)*ld + s];  B : [(2nj*nj)][ld] likewise
 *   qdd : [nj][ld] or NULL -- the nominal forward-dynamics acceleration M^-1 (u - h), a by-product. */
RBM_API int rbm_linearize_f64(const rbm_model* m, const double* q, const double* qd, const double* u, double dt, double eps, int centered,
                      double* A, double* B, double* qdd, int64_t n, int64_t ld, void* stream);

/* The transition itself (what rbm_linearize_f64 differentiates; MuJoCo's mj_forward + Euler integration for this plant,
 * core/simulate.py:270):  qdd = M(q)^-1 (u - h(q, qd));  qd+ = qd + dt qdd;  q+ = q + dt qd+.
 *   q, qd : [nj][ld];  u : [nj][ld] or NULL = zeros;  qdd : [nj][ld] or NULL;  q_next, qd_next : [nj][ld] or both NULL
 * (q_next / qd_next may alias q / qd: every sample is read before it is written). */
RBM_API int rbm_forward_dynamics_f64(const rbm_model* m, const double* q, const double* qd, const double* u, double dt, double* qdd, double* q_next,
                             double* qd_next, int64_t n, int64_t ld, void* stream);

/* ---- closed-loop replay (reference core/simulate.py:185-270), n environments per launch, one per thread ---------------
 * The reference's main loop with mj_step replaced by the transition above.  Per step: tgt = plan(step) (quintic profile as in
 * rbm_rnea_planned_*), tgt_ctrl = ID(tgt) (:187-188); act = (qpos, qvel, qacc of the PREVIOUS forward pass) (:191-194);
 * res = [(tgt_q - qpos) / pos_residual_divisor, tgt_qd - qvel] (mj_differentiatePos is called with m.nu in its dt slot: pass nu
 * = 6 to replay the reference, 1 for the plain difference) (:257-265);  ctrl = tgt_ctrl - gain res (:268);  forward pass + semi-
 * implicit Euler (:270).  On frame steps (`frame_count <= time * fps`, :196) a record
 *   [act (3 nj) | V_s (6) | dV_s (6) | wrench (6)]
 * is written: sensor-frame twists of act (:202-209) and the F/T reading left by the previous forward pass (:218-221), modelled
 * as the Newton-Euler wrench Y(V_s, dV_s) phi_sensed of the sensed subtree (MuJoCo: cfrc_int of the site's body).  The loop
 * starts from one forward pass at (q0, qd0) with ctrl = 0.
 *   plan_coeffs (6), displacement (nj), pos_offset (nj): HOST;  gain [nj][2 nj] row-major, phi_sensed (10): DEVICE
 *   q0, qd0 (or NULL = rest): [nj][ld] device;  frames: [max_frames][3 nj + 18][ld] device (frames beyond max_frames are dropped)
 *   frame_steps [max_frames], n_frames [1]: device int32 or NULL;  final_state [3 nj][ld] (qpos, qvel, qacc) or NULL */
RBM_API int rbm_closed_loop_f64(const rbm_model* m, const double* plan_coeffs, const double* displacement, const double* pos_offset, double plan_timestep,
                        double init_step, int64_t n_steps, const double* gain, const double* phi_sensed, double dt, double fps,
                        double pos_residual_divisor, const double* q0, const double* qd0, double* frames, int64_t max_frames, int32_t* frame_steps,
                        int32_t* n_frames, double* final_state, int64_t n, int64_t ld, void* stream);

/* ---- frame algebra helpers, batched (device pointers, AoS) ----------------------------------------------
 * transfer_simat (dynamics/dynamics.py:72-106): out[s] = Ad(T_s^-1)^T G_s Ad(T_s^-1); poses [n][12], simats [n][36]. */
RBM_API int rbm_transfer_simat_f64(const double* poses_Rt, const double* simats, double* out, int64_t n, void* stream);
/* coordinate_transfer_simat (dynamics.py:260-263): out[s] = Ad(T_s) G_s Ad(T_s)^T. */
RBM_API int rbm_coordinate_transfer_simat_f64(const double* poses_Rt, const double* simats, double* out, int64_t n, void* stream);
/* coordinate_transfer_imat (dynamics.py:252-257): out[s] = R I R^T + m (|t|^2 1 - t t^T); imats [n][9], mass [n]. */
RBM_API int rbm_coordinate_transfer_imat_f64(const double* poses_Rt, const double* imats, const double* mass, double* out, int64_t n, void* stream);
/* get_spatial_inertia_matrix (dynamics.py:49-69): mass [n], diag [n][3] -> [n][36]. */
RBM_API int rbm_spatial_inertia_f64(const double* mass, const double* diag, double* out, int64_t n, void* stream);
/* compose / tq2se3 / tr2se3 (transformations/transformations.py:8-50): trans [n][3] + rot [n][rot_len] (rot_len 4: wxyz
 * quaternion, 9: row-major rotation matrix) -> poses [n][12]; status [n] (device int32): 0 ok, 1 non-unit quaternion,
 * 2 invalid rotation matrix (the conditions under which liegroups raises ValueError). */
RBM_API int rbm_compose_f64(const double* trans, const double* rot, int rot_len, double* poses_Rt, int32_t* status, int64_t n, void* stream);
/* extract_linvel / extract_linacc_frame_transferred (dynamics.py:160-212): twists, dtwists [n][6], points [n][3] ->
 * linvel, linacc [n][3] (either output may be NULL; dtwists may be NULL when linacc is). */
RBM_API int rbm_point_motion_f64(const double* twists, const double* dtwists, const double* points, double* linvel, double* linacc, int64_t n,
                         void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RBM_B200_H */
