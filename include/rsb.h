/* rsb.h -- C-ABI of the B200-native batched rigid-body step ("raisim batch").
 *
 * This is the drop-in boundary for the hot path raisim::World::integrate() =
 * integrate1() + integrate2() and the ArticulatedSystem state/force/PD accessors around it
 * (SURVEY.md section 8b).  The reference exposes that path as C++ classes, not a plugin ABI, and the
 * reference snapshot holds none of the headers (/root/reference/.SUBMODULES.json:2 records
 * "bytes": 0; the only consumer build recorded is /root/reference/.travis.yml:11,
 * -DRAISIM_EXAMPLE=ON).  Each entry point below therefore cites the upstream *symbol* it replaces
 * ([RECALL] in SURVEY.md: include/raisim/World.hpp, object/ArticulatedSystem/ArticulatedSystem.hpp,
 * contact/Contact.hpp); the header-only facade in include/raisim/ forwards those symbols here.
 *
 * Rules: plain C, opaque handles, int status (0 = OK, negative = error, text via rsb_last_error()),
 * no exceptions across the boundary, all buffers caller-owned.  One handle <-> one host thread.
 * All batched arrays are float32; `where` says whether a caller buffer is host or device memory.
 * Device work is enqueued on the batch's stream (rsb_batch_set_stream) and is asynchronous unless a
 * host buffer is read back.
 */
#ifndef RSB_H_
#define RSB_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RSB_OK 0
#define RSB_ERR_INVALID (-1)
#define RSB_ERR_PARSE (-2)
#define RSB_ERR_CUDA (-3)
#define RSB_ERR_UNSUPPORTED (-4)

#define RSB_HOST 0
#define RSB_DEVICE 1

#define RSB_KMAX 8 /* contacts kept per environment (the deepest RSB_KMAX candidates) */
#define RSB_LMAX 4 /* joint-limit constraints kept per environment (the first RSB_LMAX violated joints) */

/* ArticulatedSystem::ControlMode */
#define RSB_FORCE_AND_TORQUE 0
#define RSB_PD_PLUS_FEEDFORWARD_TORQUE 1

typedef struct rsb_model rsb_model; /* immutable robot description (URDF -> tables) */
typedef struct rsb_batch rsb_batch; /* N environments of one model on one GPU        */

/* World::setTimeStep, setGravity, setERP, setContactSolverParam, setDefaultMaterial */
typedef struct rsb_params {
  float dt;          /* World::setTimeStep                               (default 0.0025) */
  float gravity[3];  /* World::setGravity                                (0,0,-9.81)      */
  float erp;         /* World::setERP                                    (0)              */
  float alpha_init;  /* World::setContactSolverParam(alpha_init, ...)    (1)              */
  float alpha_min;   /*                                                  (1)              */
  float alpha_decay; /*                                                  (1)              */
  int max_iter;      /*                                                  (150)            */
  float threshold;   /*                                                  (1e-6, float32)  */
  float mu;          /* World::setDefaultMaterial friction               (0.8)            */
  float restitution; /* World::setDefaultMaterial restitution            (0)              */
  float rest_threshold; /* restitution threshold velocity               (0.01)           */
  /* Stagnation exit of the Gauss-Seidel loop (NOT in the reference; stall_window = 0 restores the
   * plain maxIter behaviour): every stall_window iterations, stop if the largest impulse update has
   * not dropped below stall_ratio x its value one window earlier (then see stall_reg below).  A safety
   * net for the contact sets on which the published per-contact rule enters a limit cycle (~1 % of the
   * problems of fallen robots even with the accelerated sweeps; none of standing ones); DESIGN.md 5. */
  int stall_window;     /*                                               (8)              */
  float stall_ratio;    /*                                               (0.5)            */
  int joint_limits;     /* enforce URDF <limit lower upper> as unilateral rows of the same solve (1) */
  /* Anderson acceleration of the Gauss-Seidel sweep map (NOT in the reference; accel_m = 0 restores the plain sweeps of the
   * published method): from sweep accel_start on, the next iterate is extrapolated from the last accel_m + 1 sweep
   * outputs g_k and residuals f_k = g_k - x_k (least squares over the residual differences; history dropped when the
   * residual doubles).  Same fixed point; redundant contact sets (box feet, knee + foot on one shank) converge in a
   * third of the sweeps and quickly converging problems never reach accel_start.  DESIGN.md section 5. */
  int accel_m;          /* 0 = off, 2 = on                               (2)              */
  int accel_start;      /* first extrapolation after this sweep          (6)              */
  /* What the FIRST failed stagnation check does: with stall_reg > 0 the solve goes on with the Delassus matrix
   * G + stall_reg * mean(diag G) * I -- a slightly compliant contact set (constraint-force mixing) on which the sweeps do
   * converge -- and only a second failed check ends it; stall_reg = 0 ends it at once.  Fires on ~1 % of the steps of
   * fallen robots whose joint stops fight sticking contacts, never on standing ones (DESIGN.md section 5). */
  float stall_reg;      /*                                               (0.02)           */
} rsb_params;

/* raisim::Contact as returned by ArticulatedSystem::getContacts(): 12 words */
typedef struct rsb_contact {
  int32_t local_body;  /* Contact::getlocalBodyIndex()                                      */
  int32_t pair_index;  /* terrain feature: 0 = Ground plane, 2*cell+tri on a HeightMap     */
  float position[3];   /* Contact::getPosition()  (world)                                   */
  float normal[3];     /* Contact::getNormal()    (world, terrain -> robot)                 */
  float impulse[3];    /* Contact::getImpulse()   (world, on the robot)                     */
  float depth;         /* Contact::getDepth()                                               */
} rsb_contact;

/* host-side view of the model tables (doubles; arrays owned by the model) */
typedef struct rsb_model_tables {
  int nb, nq, nv, floating, ncoll, npts;
  const int *parent, *jtype, *qidx, *vidx, *depth;
  const double *jpos, *jrot, *axis, *mass, *com, *inertia, *jlimit;
  const int *cbody, *ctype;
  const double *csize, *cpos, *crot;
  const int *pt_body, *pt_coll, *pt_feat;
  const double *pt_pos, *pt_rad;
  /* contact candidates are typed: 0 = sphere of radius pt_rad at pt_pos (radius 0: box corner / cylinder rim sample), 1 = the
   * segment pt_pos .. pt_pos2 swept by pt_rad (capsule / cylinder side), 2 = the box of collision body pt_coll against terrain
   * vertices; types 1 and 2 come after the points and act on height maps only */
  const int* pt_type;
  const double* pt_pos2;
  const double* jeffort; /* [nb] URDF <limit effort> of the joint that carries the body (1e30 = none): the commanded torque saturates there */
} rsb_model_tables;

/* zero-copy device view (rows are padded: element (env, i) of X lives at X[env * X_stride + i]) */
typedef struct rsb_device_view {
  int num_envs, nq, nv, gc_stride, gv_stride;
  float *gc, *gv, *tau_ff, *ptarget, *vtarget;
  int32_t* ncontacts;
  rsb_contact* contacts; /* [num_envs][RSB_KMAX] */
} rsb_device_view;

const char* rsb_last_error(void);
int rsb_version(void);

/* ---- model: World::addArticulatedSystem(urdf) parsing half (SURVEY 3.3) ---------------------- */
int rsb_model_create_from_urdf(const char* path_or_xml, rsb_model** out);
void rsb_model_destroy(rsb_model* m);
/* binary cache of the compiled model tables (SURVEY 8f N2): skips XML parsing for fleets of workers; same-architecture file */
int rsb_model_save(const rsb_model* m, const char* path);
int rsb_model_load(const char* path, rsb_model** out);
int rsb_model_dims(const rsb_model* m, int* nq, int* nv, int* nb, int* ncoll, int* npts);
int rsb_model_get_tables(const rsb_model* m, rsb_model_tables* out);
int rsb_model_body_index(const rsb_model* m, const char* name);    /* ArticulatedSystem::getBodyIdx   */
const char* rsb_model_body_name(const rsb_model* m, int body);
int rsb_model_collision_index(const rsb_model* m, const char* name); /* getCollisionBody("LINK/k"): k-th collision body of a link */
const char* rsb_model_joint_name(const rsb_model* m, int body);
int rsb_model_frame_index(const rsb_model* m, const char* name);   /* getFrameIdxByName (link frames) */
int rsb_model_frame(const rsb_model* m, int frame, int* body, double pos[3], double rot[9]);

/* ---- batch lifetime --------------------------------------------------------------------------- */
int rsb_batch_create(const rsb_model* m, int num_envs, int device, rsb_batch** out);
void rsb_batch_destroy(rsb_batch* b);
int rsb_batch_set_stream(rsb_batch* b, void* cuda_stream);
int rsb_batch_sync(rsb_batch* b);
int rsb_batch_num_envs(const rsb_batch* b);

/* ---- world set-up ----------------------------------------------------------------------------- */
int rsb_batch_set_ground(rsb_batch* b, float z);                                   /* World::addGround    */
int rsb_batch_set_heightmap(rsb_batch* b, int x_samples, int y_samples, float x_size, float y_size,
                            float center_x, float center_y, const float* heights_host); /* World::addHeightMap */
int rsb_batch_clear_terrain(rsb_batch* b);
/* terrain atlas: upstream gives every environment its own World, hence possibly its own HeightMap; here `count` same-sized
 * maps ([count][y_samples][x_samples], host) share one batch and map_of_env[num_envs] (host) picks one per environment */
int rsb_batch_set_heightmaps(rsb_batch* b, int count, int x_samples, int y_samples, float x_size, float y_size,
                             float center_x, float center_y, const float* heights_host, const int32_t* map_of_env);
int rsb_batch_set_params(rsb_batch* b, const rsb_params* p);
int rsb_batch_get_params(const rsb_batch* b, rsb_params* p);
int rsb_params_default(rsb_params* p);
/* friction of one collision body (index in rsb_model_tables order) against the terrain; mu < 0 = default material.
 * The per-body half of World::setMaterialPairProp / getCollisionBody(name).setMaterial */
int rsb_batch_set_collision_friction(rsb_batch* b, int collision_body, float mu);

/* ---- state and actuation (ArticulatedSystem::setState/getState/setPdGains/setPdTarget/
 *      setGeneralizedForce/setControlMode); buffers are tight [env_count][nq|nv] float32 ---------- */
int rsb_batch_set_state(rsb_batch* b, const float* gc, const float* gv, int env_begin, int env_count, int where);
int rsb_batch_get_state(rsb_batch* b, float* gc, float* gv, int env_begin, int env_count, int where);
int rsb_batch_set_pd_gains(rsb_batch* b, const float* kp, const float* kd);        /* [nv], host, all envs */
int rsb_batch_set_pd_target(rsb_batch* b, const float* ptarget, const float* vtarget, int env_begin, int env_count, int where);
/* zero-copy PD targets for trainers on the same GPU: the step kernel reads rows [env][0..nq) straight from the
 * caller's device buffer (row_stride floats apart) until targets are copied in again or NULL is bound */
int rsb_batch_bind_pd_target(rsb_batch* b, const float* ptarget_device, int row_stride);
int rsb_batch_set_generalized_force(rsb_batch* b, const float* tau, int env_begin, int env_count, int where);
int rsb_batch_set_control_mode(rsb_batch* b, int mode);
/* ArticulatedSystem::setExternalForce(bodyIdx, pos, force) / setExternalTorque(bodyIdx, torque): one wrench per
 * environment on `body`, applied at point_body[3] (body frame, host pointer; NULL = body origin); force / torque are
 * [env_count][3] world-frame rows (NULL = zero).  Like upstream it acts during the next integrate() call only (all fused
 * sub-steps of that call) and is cleared afterwards. */
int rsb_batch_set_external_wrench(rsb_batch* b, int body, const float* force, const float* torque, const float* point_body,
                                  int env_begin, int env_count, int where);
/* ArticulatedSystem::getGeneralizedForce(): feed-forward + PD force applied over the last integrate() */
int rsb_batch_get_generalized_force(rsb_batch* b, float* tau, int env_begin, int env_count, int where);

/* ---- the hot path: World::integrate1(), integrate2(), integrate() ----------------------------- */
int rsb_batch_integrate1(rsb_batch* b);               /* kinematics, collision, M, h (for the getters)   */
int rsb_batch_integrate2(rsb_batch* b);               /* contact solve + state integration               */
int rsb_batch_integrate(rsb_batch* b, int substeps);  /* substeps x integrate(), one fused launch        */

/* ---- read-backs (lazy getters of the reference, SURVEY 3.4): M, h and poses always describe the current state ---- */
int rsb_batch_get_mass_matrix(rsb_batch* b, int env_begin, int env_count, float* out, int where);     /* [n][nv*nv] getMassMatrix     */
int rsb_batch_get_nonlinearities(rsb_batch* b, int env_begin, int env_count, float* out, int where);  /* [n][nv]    getNonlinearities */
int rsb_batch_get_body_poses(rsb_batch* b, int env_begin, int env_count, float* rot, float* pos, int where); /* [n][nb*9],[n][nb*3] */
int rsb_batch_get_contacts(rsb_batch* b, rsb_contact* out, int32_t* counts, int env_begin, int env_count, int where); /* out [n][RSB_KMAX] */
int rsb_batch_get_contact_points(rsb_batch* b, int32_t* pt_index, int env_begin, int env_count, int where);          /* [n][RSB_KMAX] candidate-point ids */
int rsb_batch_get_solver_iterations(rsb_batch* b, int32_t* iters, int env_begin, int env_count, int where);          /* getContactSolver().getLoopCounter() */
int rsb_batch_get_diverged(rsb_batch* b, int32_t* flags, int env_begin, int env_count, int where);                   /* 1 = state went non-finite in the last step: reset it */
/* how the last contact solve of every environment ended */
#define RSB_SOLVER_CONVERGED 0           /* largest impulse update < threshold                                         */
#define RSB_SOLVER_CONVERGED_COMPLIANT 1 /* ... on the compliant contact set entered after a failed stagnation check   */
#define RSB_SOLVER_STALLED 2             /* ended by a failed stagnation check (second one when stall_reg > 0)          */
#define RSB_SOLVER_MAXITER 3             /* max_iter sweeps without reaching the threshold                              */
int rsb_batch_get_solver_status(rsb_batch* b, int32_t* status, int env_begin, int env_count, int where);
int rsb_batch_get_solver_residual(rsb_batch* b, float* resid, int env_begin, int env_count, int where);              /* largest impulse update of the last sweep (< threshold: converged) */
/* FK, M and h of the CURRENT state for the getters above, without touching the contact records of the last integrate()
 * (upstream's getters are lazy the same way).  The getters call it themselves when the state changed through this API;
 * call it explicitly after writing the state through rsb_batch_device_ptrs() views. */
int rsb_batch_update_kinematics(rsb_batch* b);
int rsb_batch_device_ptrs(rsb_batch* b, rsb_device_view* view);
int64_t rsb_batch_launch_count(const rsb_batch* b);   /* kernels launched by this batch so far */

/* ---- RaisimGym observation row (VectorizedEnvironment::observe), ANYmal locomotion layout:
 *      [z, R^T e_z (3), joint q (nq-7), R^T v (3), R^T w (3), joint rates (nv-6)]  -> ob_dim = nq+nv-3 -- */
int rsb_batch_ob_dim(const rsb_batch* b);
int rsb_batch_observe(rsb_batch* b, float* obs, int env_begin, int env_count, int where);
/* VectorizedEnvironment::step() for the whole batch in one call: targets in, `substeps` fused
 * World::integrate() calls, observation rows out (either pointer may be NULL to skip that leg) */
int rsb_batch_control_step(rsb_batch* b, const float* ptarget, const float* vtarget, int where_in, int substeps, float* obs, int where_out);

/* ---- terrain sensing (height scans; World::rayTest).  The surface is the one the narrow phase collides with (Ground plane, or each
 *      environment's height map split into triangles as in DESIGN.md section 2); the robot itself is never hit.  Frame poses describe the
 *      current state: a frame on body 0 of a floating base is read from the gc rows, any other frame costs one kinematics launch when the
 *      state changed since the last one.  Pattern arrays (frames, points, frame-fixed rays) are host arrays, uploaded only when they differ
 *      from the previous call's.  Host outputs are complete on return; device outputs are ordered on the batch's stream. ---- */
typedef struct rsb_ray_hit {
  float distance;     /* t of the first crossing, +inf on a miss                                           */
  float position[3];  /* world-frame hit point (0 on a miss)                                               */
  float normal[3];    /* unit normal of the triangle hit, oriented +z (terrain -> outside); 0 on a miss    */
  int32_t pair_index; /* terrain feature: 0 = Ground plane, 2*cell+tri on a HeightMap; -1 = miss           */
} rsb_ray_hit;        /* 8 words */
/* out[e * out_stride + f * num_points + k] = z of frame f - terrain height at (p_f + Rz(yaw_f) [x_k, y_k]), yaw_f = atan2(R10, R00) of
 * the frame's world rotation; points off the map take the height of the nearest border point.  frames[num_frames]
 * (rsb_model_frame_index) and points_xy[num_points][2] are host arrays; out is `where` memory, out_stride >= num_frames * num_points
 * (a trainer may write the scan into columns of a wider buffer it owns: the other columns are left as they are). */
int rsb_batch_height_scan(rsb_batch* b, const int32_t* frames, int num_frames, const float* points_xy, int num_points,
                          float* out, int out_stride, int env_begin, int env_count, int where);
/* Rays o + t d/|d|, t in [0, length]: the first crossing of the terrain from either side.
 * num_frames >= 1: origins / dirs [num_rays][3] (host) are fixed in each frame (rotated with its full world rotation);
 *                  out [env_count][num_frames][num_rays].
 * num_frames == 0: origins / dirs [env_count][num_rays][3] are world-frame rays in `where` memory; out [env_count][num_rays].
 * A zero direction is an error for host arrays; a zero direction read from device memory gives a miss.  No terrain: all misses. */
int rsb_batch_ray_test(rsb_batch* b, const int32_t* frames, int num_frames, const float* origins, const float* dirs, int num_rays,
                       float length, rsb_ray_hit* out, int env_begin, int env_count, int where);

/* ---- terrain generation (raisim::TerrainProperties, World::addHeightMap(centerX, centerY, terrainProperties)) ------ */
typedef struct rsb_terrain_properties {
  int x_samples, y_samples;      /* TerrainProperties::xSamples, ySamples */
  double x_size, y_size;         /* xSize, ySize [m]                       */
  double frequency;              /* base frequency of the noise [1/m]      */
  double z_scale;                /* zScale                                 */
  int fractal_octaves;           /* fractalOctaves                         */
  double fractal_lacunarity;     /* fractalLacunarity                      */
  double fractal_gain;           /* fractalGain                            */
  double step_size;              /* stepSize (0 = smooth)                  */
  double height_offset;          /* heightOffset                           */
  uint32_t seed;                 /* seed                                   */
} rsb_terrain_properties;
int rsb_terrain_generate(const rsb_terrain_properties* p, float* heights_out /* [y_samples][x_samples] */);

/* height-map files: World::addHeightMap(raisimHeightMapFileName, centerX, centerY) -- text, header "xSamples ySamples xSize
 * ySize" then the heights, x fastest -- and World::addHeightMap(pngFileName, centerX, centerY, xSize, ySize, heightScale,
 * heightOffset) -- 8/16-bit PNG, height = pixel * scale + offset.  heights == NULL only reports the sample counts. */
int rsb_heightmap_read_text(const char* path, int* x_samples, int* y_samples, double* x_size, double* y_size, float* heights, int capacity);
int rsb_heightmap_read_png(const char* path, double height_scale, double height_offset, int* x_samples, int* y_samples, float* heights, int capacity);

/* ---- multi-GPU inside one process (SURVEY 8e): one rsb_batch per GPU, NCCL all-gather of the observation rows ----
 *      (NCCL is bound at run time; bench.py uses torch.distributed for the same collective, one process per GPU) */
typedef struct rsb_comm rsb_comm;
int rsb_comm_init(rsb_batch** batches, int ndev, rsb_comm** out);             /* ncclCommInitAll over the batches' devices */
int rsb_comm_allgather_obs(rsb_comm* c, float* const* obs_all_per_device);     /* observe + ncclAllGather on every device     */
void rsb_comm_destroy(rsb_comm* c);

/* ---- multi-GPU, one process per GPU: the observation all-gather FUSED into the step kernel over NVLink peer memory ----
 * Every rank allocates two gathered-rows buffers [world * num_envs][ob_dim] and one counter row unsigned[world]
 * (rsb_peer_buffer_create: cudaMalloc + CUDA IPC handle), ships the 64-byte handles to its peers over any host channel
 * (torch.distributed / MPI / a pipe), maps theirs (rsb_peer_buffer_open) and hands all pointers to its batch.  From then on
 * a control step that returns observation rows on the device also stores every finished row straight into every rank's
 * buffer (parity = control step & 1) while the kernel is still running, and bumps a counter on every rank as each CTA ends;
 * the last CTA of the launch stays until every rank's counter shows its rows of this step, so the launch completes when the
 * gathered rows are complete (bounded: a dead peer traps).  rsb_batch_wait_observation_peers() tells which of the two buffers
 * holds the rows of the last step.  No NCCL call on the data path.  Every rank must step the same number of times. */
int rsb_peer_buffer_create(int device, size_t bytes, void** dev_ptr, unsigned char* handle64 /* may be NULL */);
int rsb_peer_buffer_open(int device, const unsigned char* handle64, void** dev_ptr);
int rsb_peer_buffer_close(void* dev_ptr);
int rsb_peer_buffer_destroy(void* dev_ptr);
int rsb_batch_set_observation_peers(rsb_batch* b, int world, int rank, void* const* obs_all /* [2 * world] */, void* const* flags /* [world] */);
int rsb_batch_wait_observation_peers(rsb_batch* b, int* buffer_parity /* may be NULL */);

/* ---- RaisimGym task on the device (raisimGymTorch VectorizedEnvironment.hpp / envs/rsg_anymal/Environment.hpp,
 *      [RECALL]): pTarget = action * std + mean; reward = torque_coeff * |tau|^2 + forward_vel_coeff * min(4, v_body_x);
 *      an episode terminates on any contact whose local body is not in foot_bodies (reward += terminal_reward, state reset) -- */
int rsb_batch_gym_configure(rsb_batch* b, const float* gc_init, const float* gv_init, const float* action_mean, const float* action_std,
                            const int32_t* foot_bodies, int n_foot, float torque_coeff, float forward_vel_coeff, float terminal_reward);
int rsb_batch_gym_reset(rsb_batch* b);                                             /* VectorizedEnvironment::reset() */
/* ::step() + ::observe() in ONE launch of the step kernel: action rows -> PD targets, `substeps` x World::integrate(), reward,
 * isTerminalState(), reset() of the terminated environments, observation rows of the resulting state.  Needs rsb_batch_set_pd_gains(). */
int rsb_batch_gym_step(rsb_batch* b, const float* action, int where_in, int substeps, float* obs, float* reward, unsigned char* done,
                       int where_out);

#ifdef __cplusplus
}
#endif
#endif /* RSB_H_ */
