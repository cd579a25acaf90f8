/* softgrip.h -- C-ABI of libsoftgrip.so, the B200-native batched replacement for the MuJoCo step
 * loop that the reference's ManEnv drives through mujoco-py.
 *
 * The reference has no FFI layer of its own for this path: its binding is mujoco-py's Cython module,
 * and ManEnv touches exactly these entry points of it (ref: environment/manenv.py, line numbers below).
 * Each function here names the mujoco-py / MuJoCo call it replaces.
 *
 * Conventions
 *   - every function returns 0 on success, <0 on error; sg_last_error() gives a thread-local message;
 *   - a world that diverges (NaN / |x|>1e10, MuJoCo's mj_checkPos/Vel/Acc) is reset in place and the
 *     event is DATA (status bits per world), never an error return;
 *   - "dev" pointers are CUDA device pointers on the batch's device, "host" pointers are host memory;
 *   - per-world layouts are world-major: state [W][nv], sensors [W][nsensordata],
 *     trajectories [W][T][nsensordata] (one world's rows are contiguous = the reference's (T,12) sample);
 *   - real-valued *inputs* (parameters, ctrl, state) are always fp64; *outputs* produced by the kernels
 *     (sensor rows, trajectories) are in the batch precision: float for precision 32, double for 64;
 *   - a batch is not thread-safe; all work is enqueued on the cudaStream_t given as `stream`
 *     (NULL = legacy default stream) and is asynchronous unless stated otherwise.
 */
#ifndef SOFTGRIP_H
#define SOFTGRIP_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct sg_model sg_model;   /* compiled model (host + device constant tables)  */
typedef struct sg_batch sg_batch;   /* W independent worlds of one model on one device */

/* per-world status bits (sg_batch_status) */
#define SG_ST_DIVERGED    1   /* state was reset by the NaN/1e10 check (ref: manenv.py:50-51 MujocoException path) */
#define SG_ST_CON_FULL    2   /* contact capacity exceeded, extra contacts dropped (MuJoCo: nconmax warning)     */
#define SG_ST_EFC_FULL    4   /* reserved                                                                       */
#define SG_ST_UNSUPPORTED 8   /* a geom pair outside the restated narrowphase set overlapped (box-box, plane-box) */

typedef struct sg_info {
  int nv;             /* dofs = finger hinges + shell sliders                */
  int nfinger;        /* finger (hinge) dofs                                 */
  int nshell;         /* shell sliders of the composite object               */
  int neq;            /* equality constraints (fix + neighbour + tendon)     */
  int nu;             /* actuators / ctrl entries                            */
  int nsensordata;    /* sensor row length (12 for the reference gripper)    */
  int nlevels;        /* Gauss-Seidel dependency levels of the equality block */
  int maxcon;         /* per-world contact capacity                          */
  int smem_bytes32;   /* dynamic shared memory per world, fp32 build         */
  int smem_bytes64;   /* dynamic shared memory per world, fp64 build         */
  int ngeom;
  int reserved[5];
} sg_info;

/* Episode schedule of sg_batch_rollout: the ctrl protocol of create_dataset.log_into_file
 * (ref: create_dataset.py:33-60).  Env-step t (0 <= t < nrows) runs `sim_step` physics steps and then
 * records one sensor row.  Before executing env-step t, if ctrl_event[t] != 0 the ctrl vector is set to
 * ctrl_value[t*nu .. t*nu+nu-1] (close_hand / toggle_grip, ref: manenv.py:87-101). */
typedef struct sg_schedule {
  int sim_start;              /* physics steps run by reset() before recording (ref: manenv.py:60-61) */
  int sim_step;               /* physics steps per env-step (ref: manenv.py:44-49)                     */
  int nrows;                  /* env-steps = recorded rows (200 in the reference)                      */
  const int* ctrl_event;      /* host, [nrows]                                                         */
  const double* ctrl_value;   /* host, [nrows][nu]                                                     */
} sg_schedule;

const char* sg_last_error(void);
int sg_version(void);

/* replaces mujoco_py.load_model_from_path (ref: manenv.py:27,36): takes the blob produced by the MJCF
 * compiler (soft-grip_b200/mjcf.py) and builds the device plan (tables, Gauss-Seidel level schedule). */
int sg_model_load(const void* blob, size_t nbytes, sg_model** out);
int sg_model_info(const sg_model* m, sg_info* out);
void sg_model_destroy(sg_model* m);

/* replaces mujoco_py.MjSim(model) (ref: manenv.py:28,37) for `nworlds` worlds. precision: 32 or 64. */
int sg_batch_create(const sg_model* m, int nworlds, int device, int precision, sg_batch** out);
void sg_batch_destroy(sg_batch* b);
int sg_batch_nworlds(const sg_batch* b);
int sg_batch_precision(const sg_batch* b);

/* replaces the writes to sim.model.jnt_stiffness[joint_ids] / tendon_stiffness[tendon_ids]
 * (ref: manenv.py:103-109).  joint_mask: host, [nv] ints, 1 where the per-world stiffness applies;
 * tendon0: whether it also applies to tendon 0 (the composite's volume tendon). */
int sg_model_set_stiffness_targets(sg_model* m, const int* joint_mask, int tendon0);
/* per-world parameters, dev fp64 arrays of length W (objoff: [W][3]); NULL keeps the model value.
 * stiffness -> masked shell joints (+ tendon 0); damping -> all shell joints (extension, not in the
 * reference); tdamping -> tendon 0 damping (extension); objoff -> translation of the object body. */
int sg_batch_set_params(sg_batch* b, const double* stiffness, const double* damping,
                        const double* tdamping, const double* objoff, void* stream);
/* per-geom name bitmask for the contact flag of get_sensor_sensordata (ref: manenv.py:65-83):
 * bit0 = geom name contains obj_name, bit(1+k) = contains finger_names[k]. host, [ngeom]. */
int sg_model_set_geom_mask(sg_model* m, const int* mask);

/* replaces sim.reset() == mj_resetData (ref: manenv.py:57) for every world */
int sg_batch_reset(sg_batch* b, void* stream);
/* replaces sim.data.ctrl[i] = v (ref: manenv.py:95,100). ctrl: dev fp64 [W][nu] */
int sg_batch_set_ctrl(sg_batch* b, const double* ctrl, void* stream);
/* same, one host vector [nu] broadcast to all worlds */
int sg_batch_set_ctrl_all(sg_batch* b, const double* ctrl_host, void* stream);
/* replaces sim.forward() == mj_forward (ref: manenv.py:58): refreshes sensor rows without integrating */
int sg_batch_forward(sg_batch* b, void* sens_out, int* touch_out, void* stream);
/* replaces `for _ in range(nsub): sim.step()` + the sensordata/contact read-out
 * (ref: manenv.py:44-53,65-85). sens_out: dev [W][nsensordata] (batch precision) or NULL;
 * touch_out: dev [W] ints or NULL (OR over contacts with an object geom of (mask>>1)). */
int sg_batch_step(sg_batch* b, int nsub, void* sens_out, int* touch_out, void* stream);
/* whole episode in one launch; state stays on-chip for the full horizon.
 * traj_out: dev [W][nrows][nsensordata] (batch precision); touch_out: dev [W][nrows] ints or NULL. */
int sg_batch_rollout(sg_batch* b, const sg_schedule* s, void* traj_out, int* touch_out, void* stream);
/* rollout through HOST buffers (what a ctypes/cgo caller without device memory uses): copies
 * stiffness_host [W] fp64 to the device, runs the episode, copies the trajectory back, synchronises.
 * traj_host: [W][nrows][nsensordata] in batch precision; touch_host/status_host may be NULL. */
int sg_batch_rollout_host(sg_batch* b, const sg_schedule* s, const double* stiffness_host,
                          void* traj_host, int* touch_host, int* status_host);

/* the same with every per-world parameter of sg_batch_set_params coming from HOST memory (fp64, [W]; objoff [W][3];
 * NULL keeps what the batch holds): BASELINE.json configs[2] randomises stiffness, damping and object pose per world */
int sg_batch_rollout_host_params(sg_batch* b, const sg_schedule* s, const double* stiffness_host,
                                 const double* damping_host, const double* tdamping_host, const double* objoff_host,
                                 void* traj_host, int* touch_host, int* status_host);
/* trajectory layout written by sg_batch_rollout (the host variants always return the world-major one):
 * SG_TRAJ_WORLD_MAJOR [W][nrows][nsensordata] -- one world's rows are contiguous = the reference's (T,12) sample
 * (ref: create_dataset.py:62-63), each row written as 128-bit vectors;
 * SG_TRAJ_SOA [nrows][nsensordata][W] -- structure of arrays, world index fastest (SURVEY section 8b `rollout`). */
#define SG_TRAJ_WORLD_MAJOR 0
#define SG_TRAJ_SOA 1
int sg_batch_set_traj_layout(sg_batch* b, int layout);

/* state access for parity tests on identical initial states (host fp64, synchronous).
 * qpos,qvel,qacc_warmstart: [W][nv]; act: [W][nu]; any pointer may be NULL. */
int sg_batch_get_state(sg_batch* b, double* qpos, double* qvel, double* act, double* qacc_warmstart);
int sg_batch_set_state(sg_batch* b, const double* qpos, const double* qvel, const double* act,
                       const double* qacc_warmstart);
/* status bits per world: host [W] ints (synchronous); clear!=0 zeroes them afterwards */
int sg_batch_status(sg_batch* b, int* status_host, int clear);
int sg_batch_sync(sg_batch* b, void* stream);

/* diagnostics of the last physics step of one world (synchronous, host fp64): key is one of
 * "qacc","qacc_smooth","ncon","nefc","solver_iter","con_dist","con_pos","con_frame","efc_force",
 * "efc_aref","efc_R"; "sweep_schedule" / "pair_runs" return the host-side step tables of the equality sweep / the
 * candidate pair list and its run-length form instead (layouts in sg_api.cu); "tensor_memory" returns how the launch
 * geometry of this batch stores the solver's working set: [tensor-memory columns per CTA (0: equality rows in shared
 * memory), columns per warp, 1 if the contact records go through the shared-memory ring].
 * Returns the element count (<0 on error); writes at most cap values.
 * The per-step keys are only valid after sg_batch_set_debug_world(b, w) and a subsequent step/forward; the table keys
 * ("sweep_schedule", "pair_runs", "tensor_memory") at any time. */
int sg_batch_set_debug_world(sg_batch* b, int world);
int sg_batch_debug_get(sg_batch* b, const char* key, double* out, int cap);

/* launch geometry chosen for this batch (host ints, out[8]): [0] lanes per world, [1] warps per CTA, [2] worlds per CTA,
 * [3] resident CTAs per SM, [4] dynamic shared memory per CTA (bytes), [5] shared memory per world (bytes),
 * [6] 0 (was: team mode, removed), [7] kernel generation (always 2: sg_step_kernel2).
 * No reference counterpart: it only documents how the worlds were packed onto the SMs (bench.py reports it). */
int sg_batch_config(const sg_batch* b, int* out);

/* development aid, no reference counterpart: SM-clock cycles per phase of the step kernel, summed over the warps of
 * all launches since the last call (out[n], n <= 16: gripper, collide, rows, warm start, solver set-up, equality
 * sweeps, limit/contact sweeps, sensors, Euler, other).  Only for batches created with SOFTGRIP_PROF=1 in the
 * environment; otherwise an error.  Returns the number of phases. */
int sg_batch_prof_get(sg_batch* b, unsigned long long* out, int n);

/* number of kernel launches issued by this batch since creation (bench.py's gpu_launches) */
long long sg_batch_launch_count(const sg_batch* b);

/* ---- the trajectory buffer downstream of the step path (SURVEY section 8 rows f1 / f4) -----------------------------
 * `traj` is [nrows][nchan] in `precision` (32: float, 64: double) on `device`, 16-byte aligned, nchan a multiple of 4
 * (<= 64): a rollout's [W][T][12] buffer with nrows = W*T.  All calls are asynchronous on `stream`. */

/* replaces functions/optimization.py:6-14 `noised_modality`: channels [0, nacc) += N(0, sigma_acc), channels
 * [nacc, nchan) += N(0, sigma_gyro) (reference: nacc 6, 0.7, 0.06), traj_out may alias traj_in.  The draws are
 * Philox4x32-10(key = seed, counter = global element index / 4) + Box-Muller in fp32, i.e. a function of (seed, element
 * index) only; first_row is the row index of traj_in[0] inside the whole dataset tensor (0 for a whole tensor), so that
 * shards noised separately -- per launch, per GPU -- equal the corresponding rows of the tensor noised in one call.  mean/std (dev fp64 [nchan], both or neither): fused standardisation out = (x + noise - mean) / std of
 * functions/optimization.py:38. */
int sg_traj_add_noise(const void* traj_in, void* traj_out, long long nrows, long long first_row, int nchan, int nacc,
                      double sigma_acc, double sigma_gyro, unsigned long long seed, const double* mean, const double* std,
                      int precision, int device, void* stream);
/* replaces `np.mean(train_x, axis=(0, 1))` / `np.std(train_x, axis=(0, 1))` of functions/utils.py:39-40 (population
 * standard deviation).  mean_out/std_out: dev fp64 [nchan]; workspace: dev, at least sg_traj_stats_workspace_bytes().
 * fp64 accumulation in a fixed order: the result is bit-reproducible for a given shape and device. */
int sg_traj_channel_stats(const void* traj, long long nrows, int nchan, int precision, int device, double* mean_out,
                          double* std_out, void* workspace, long long workspace_bytes, void* stream);
long long sg_traj_stats_workspace_bytes(long long nrows, int nchan, int device);
/* replaces `if args.mask_contact and not contact: readings = np.zeros_like(readings)` (ref: create_dataset.py:43-44,
 * 57-58) for a whole rollout: traj [nworlds][nrows_per_world][nchan] in place, touch dev [nworlds][nrows_per_world] as
 * written by sg_batch_rollout (finger-group bits of the row's object contacts, any_bit set when ncon >= 1).
 * mode 0 "intended": a row is kept iff (touch & all_fingers) == all_fingers.  mode 1 "reference-literal"
 * (ref: manenv.py:65-83 with its aliased class-level finger list): while fingers are left the flag is "all fingers seen
 * so far", afterwards "ncon >= 1"; fingers_left (dev [nworlds] ints, in/out, NULL = every episode starts with the full
 * list and nothing is carried) holds the finger bits not yet seen. */
int sg_traj_mask_contact(void* traj, const int* touch, int nworlds, int nrows_per_world, int nchan, int all_fingers,
                         int any_bit, int mode, int* fingers_left, int precision, int device, void* stream);

#ifdef __cplusplus
}
#endif
#endif
