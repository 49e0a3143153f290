/*
 * panda_b200.h -- C ABI of libpanda_b200.so: batched Panda manipulation environments on one B200.
 *
 * The reference has no FFI of its own on this path: its step is Python calling the pybullet C extension
 * (reference panda_gym/pybullet.py:34-55).  This library is what a maintainer binds instead; each entry point names
 * the reference interface it replaces.  INTEGRATION.md shows the ctypes stub.
 *
 * Conventions: every function returns 0 on success and a negative code on error (text via pg_last_error()).
 * Unless a name ends in _host, every pointer is a DEVICE pointer owned by the caller, arrays are row-major
 * [num_envs, dim], and the work is enqueued asynchronously on `stream` (a cudaStream_t passed as void*, NULL = the legacy
 * default stream).  A handle owns its SoA state in HBM, is bound to one device and is not thread-safe.
 * There is no CPU fallback: without a CUDA device pg_create fails with PG_ERR_CUDA.
 */
#ifndef PANDA_B200_H
#define PANDA_B200_H
#ifdef __cplusplus
extern "C" {
#endif

enum { PG_TASK_REACH = 0, PG_TASK_PUSH = 1, PG_TASK_SLIDE = 2, PG_TASK_PICK_AND_PLACE = 3, PG_TASK_STACK = 4, PG_TASK_FLIP = 5,
       PG_TASK_BARE = 6 /* handles made by pg_create_bare: the sim facade without a task */ };
enum { PG_CTRL_EE = 0, PG_CTRL_JOINTS = 1 };          /* panda_gym/envs/robots/panda.py:21-33 control_type */
enum { PG_REWARD_SPARSE = 0, PG_REWARD_DENSE = 1 };   /* panda_gym/envs/tasks/reach.py:60-65 reward_type */
enum { PG_F32 = 0, PG_F64 = 1 };
enum { PG_OK = 0, PG_ERR_ARG = -1, PG_ERR_CUDA = -2, PG_ERR_STATE = -3 };

typedef struct pg_env pg_env;

/* Replaces PandaXxxEnv.__init__ (panda_gym/envs/panda_tasks.py:14-113: PyBullet + Panda at (-0.6,0,0) + task scene) for
 * num_envs environments.  precision: PG_F32 (product path) or PG_F64 (parity debugging).  seed + env_id_offset key the
 * device RNG by GLOBAL environment index, so a sharded run reproduces the unsharded one.  All envs start reset.  *out is written
 * only on success; after an error it is left as it was and nothing the call allocated is kept. */
int pg_create(int task, int control_type, int reward_type, int num_envs, int device, unsigned long long seed,
              long long env_id_offset, int precision, pg_env** out);
/* The reference's sim facade used WITHOUT a task (panda_gym/pybullet.py:16-68: PyBullet() + loadURDF :510-529 + create_box / create_cylinder
 * :531-719 + create_table / create_plane :726-771), as its own tests do (test/pybullet_test.py:56-65,110-265): num_envs identical
 * worlds holding the Panda at robot_base (NULL: no robot), n_bodies <= 2 free bodies -- HOST rows
 * [shape (0 box, 1 z-cylinder), hx, hy, hz (half extents; cylinder: r, r, h/2), mass, lateral friction, pos3, quat4 (x,y,z,w)] --,
 * an optional table top at z = 0 over table_rect = {x0, x1, y0, y1} (HOST, NULL: none) and an optional ground plane at *ground_z
 * (HOST, NULL: none).  Joints start at 0 with the velocity motors loadURDF leaves (target 0, max impulse 1 per sub-step).
 * Such a handle is advanced with pg_sim_step and driven with pg_set_motors; pg_get_state / pg_set_state / pg_get_link_state /
 * pg_inverse_kinematics_link / snapshots work as on task handles (state rows without a goal).  *out is written only on success, as
 * with pg_create. */
int pg_create_bare(int num_envs, int device, int precision, const double* robot_base, int n_bodies, const double* bodies,
                   const double* table_rect, const double* ground_z, pg_env** out);
/* PyBullet.control_joints -> setJointMotorControlArray (pybullet.py:462-477), per world: DEVICE rows [N, 9, 5] =
 * {position gain, velocity gain, target angle, target velocity, max force} for joints 0-6, 9, 10 (POSITION_CONTROL as the
 * reference issues it: 0.1, 1.0, target, 0, force).  mask (DEVICE, NULL = all) selects the worlds that are written. */
int pg_set_motors(pg_env* env, const double* motors, const unsigned char* mask, void* stream);
int pg_get_motors(pg_env* env, double* motors, void* stream);
/* PyBullet.step (pybullet.py:52-55): n_substeps x stepSimulation of a bare world with its current motors. */
int pg_sim_step(pg_env* env, int n_substeps, void* stream);
int pg_destroy(pg_env* env);                                            /* RobotTaskEnv.close, core.py:291-292 */
/* observation / goal / action widths and the TimeLimit length (panda_gym/__init__.py:18,46) */
int pg_dims(const pg_env* env, int* obs_dim, int* goal_dim, int* action_dim, int* max_episode_steps, int* state_dim);

/* RobotTaskEnv.reset (core.py:240-250) for the envs whose mask byte is non-zero (NULL = all): neutral joints, zero
 * velocities, goal and object placement either sampled on the device (distributions of tasks/<task>.py _sample_goal /
 * _sample_object) or taken from goal_override [N,G] / object_override [N,3*n_objects] (float64; NULL = sample).
 * seeds [N] uint64 (DEVICE) is RobotTaskEnv.reset(seed=k) batched (core.py:240-244: the task RNG is re-created from the seed):
 * each reset env's draws are keyed by ITS seed alone, so equal seeds give equal goals / object placements in any env of any handle
 * (reference test/seed_test.py); NULL keys them by the handle's seed, the global env index and the episode.  The draws come from
 * the device's Philox stream, not numpy's PCG64 -- the single-env facade reproduces the reference's seeded values bit-for-bit on
 * the host and injects them through the overrides.
 * Writes obs/ag/dg rows of the reset envs only (any of them may be NULL). */
int pg_reset(pg_env* env, const unsigned char* mask, const unsigned long long* seeds, const double* goal_override,
             const double* object_override, float* obs, float* achieved_goal, float* desired_goal, void* stream);
/* The task constructors' keyword arguments (tasks/reach.py:15-23 distance_threshold, goal_range; push.py:12-25; slide.py:12-27;
 * pick_and_place.py:13-29; stack.py:11-25; flip.py:13-24) as kernel parameters: the success / sparse-reward threshold used inside
 * pg_step, the goal noise box [low, high] (3 doubles each, HOST; what the reference builds from goal_range / goal_xy_range /
 * goal_z_range / goal_x_offset) and the object xy noise box (2 doubles each; obj_xy_range).  NULL keeps a range.  Takes effect
 * from the next reset / step. */
int pg_set_task_params(pg_env* env, double distance_threshold, const double* goal_range_low, const double* goal_range_high,
                       const double* obj_range_low, const double* obj_range_high);
/* PyBullet(n_substeps=...) (pybullet.py:26,39,52-55): stepSimulation calls per env step (default 20). */
int pg_set_substeps(pg_env* env, int n_substeps);

/* RobotTaskEnv.step (core.py:280-289) for every env: Panda.set_action (panda.py:52-70), 20 x stepSimulation
 * (pybullet.py:52-55), _get_obs (core.py:229-238), is_success, compute_reward; truncated = TimeLimit.
 * auto_reset != 0: envs that terminated or truncated are reset in the same call (device-sampled goal/object) and their
 * obs/ag/dg rows hold the reset observation while reward/terminated/truncated describe the finished step.
 * target_quat [N,4] (NULL = none) is the fork's orientation-target control (panda_gym/envs/robots/panda_ori.py:52-99:
 * set_action(action, euler_xyz)): a per-env EE target quaternion (x,y,z,w; float32, normalised inside) fed to the IK instead of
 * (1,0,0,0).  ee control only (PG_ERR_ARG otherwise).
 * contacts / contact_count (NULL = no report) are pybullet getContactPoints after RobotTaskEnv.step, for every env: the contacts of
 * the step's last sub-step (rows below; normalForce = applied impulse / timeStep) and their number per env.  contacts [N, C, 16]
 * float32 with C = pg_max_contacts; rows at and beyond contact_count[i] are unspecified.  Row words:
 *   0-2 contact point (world), as the contact model generates it;  3-5 normal on B, pointing from B to A (world);  6 normal force (N);
 *   7 lateral friction force 1 (N), 8-10 its direction;  11 lateral friction force 2 (N), 12-14 its direction;  15 id_a + 32 * id_b
 *   (an exact float).  Ids are pg_render's segmentation ids: 1 plane, 2 table, 3 / 4 objects, 14 hand (link 8), 15 / 16 fingers
 *   (links 9 / 10).  There is no contactDistance.  With auto_reset the report describes the finished step, like reward.
 * Ordering: everything the call enqueues is ordered after the work already on `stream` and completes before work enqueued on
 * `stream` afterwards.  Batches of >= 4096 envs are advanced by several launches (a step cut into sub-step segments, each after a
 * re-sort of the thread -> env map) and, from 16384 envs, in env groups on streams the handle owns, forked from and joined back
 * to `stream` with events (legal under stream capture).  None of this changes a result. */
int pg_step(pg_env* env, const float* actions, const float* target_quat, float* obs, float* achieved_goal, float* desired_goal,
            float* reward, unsigned char* terminated, unsigned char* truncated, int auto_reset,
            float* contacts, unsigned char* contact_count, void* stream);
/* C of the rows above: contacts per env and sub-step of the handle's scene (10, or 22 for Stack; later candidates are dropped). */
int pg_max_contacts(const pg_env* env, int* per_env);
/* Action scaling of Panda.set_action: defaults 0.05 (ee / joint displacement, panda.py:81,103) and 0.2 (fingers, panda.py:65);
 * the fork's panda_cartesian.py:67,157 uses 1.0 / 1.0. */
int pg_set_action_scale(pg_env* env, double ee_scale, double finger_scale);
/* pg_step with HOST buffers and without orientation targets or contact report: actions are copied to the device, the step runs, all
 * outputs are copied back and the stream is synchronised before returning (the end-to-end path a CPU learner uses). */
int pg_step_host(pg_env* env, const float* actions, float* obs, float* achieved_goal, float* desired_goal, float* reward,
                 unsigned char* terminated, unsigned char* truncated, int auto_reset);

/* Page-lock a caller-owned host buffer (cudaHostRegister) so that pg_step_host copies to / from it directly instead of through the
 * handle's staging slabs; unpin before freeing the buffer.  Buffers that are not pinned work too (one extra host copy). */
int pg_host_pin(void* ptr, size_t bytes);
int pg_host_unpin(void* ptr);

/* Task.compute_reward / Task.is_success (tasks/<task>.py, utils.py:4-30) on M rows of achieved/desired goals
 * (dtype PG_F32 or PG_F64 inputs; float32 rewards, uint8 success) -- the HER relabelling entry point.  threshold is the task's
 * distance_threshold (the reference's defaults: 0.05, 0.1 for Stack, 0.2 for Flip); it is compared in the dtype of the distance, as
 * numpy does with a Python-float threshold. */
int pg_compute_reward(int task, int reward_type, double threshold, const void* achieved_goal, const void* desired_goal,
                      float* reward, long long m, int dtype, void* stream);
int pg_is_success(int task, double threshold, const void* achieved_goal, const void* desired_goal, unsigned char* success,
                  long long m, int dtype, void* stream);
/* HER relabelling fused with compute_reward (replaces the gather + env.compute_reward round trip of stable-baselines3's
 * HerReplayBuffer that reference examples/train_push.py:1-12 sets up; rewards as tasks/<task>.py compute_reward with threshold as
 * above).  next_achieved_goal and desired_goal are the replay buffer's [R, G] goal arrays (device) with a row pitch of `pitch`
 * elements (pitch >= G): a buffer that stores its goals padded to 32 bytes (pitch 8 for fp32 goals of 3, 4 or 6 components) makes
 * every gathered row exactly one DRAM sector instead of one or two.  For each of the M sampled transitions j: the new goal is
 * next_achieved_goal[goal_src[j]] (desired_goal[src[j]] when goal_src[j] < 0) and the reward is compute_reward(next_achieved_goal[src[j]],
 * new goal).  Outputs (dense): desired_goal_out [M, G], achieved_goal_out [M, G] (may be NULL), reward [M] float32. */
int pg_her_relabel(int task, int reward_type, double threshold, const void* next_achieved_goal, const void* desired_goal,
                   long long pitch, const long long* src, const long long* goal_src, void* desired_goal_out,
                   void* achieved_goal_out, float* reward, long long m, int dtype, void* stream);
/* Task.compute_reward / is_success on HOST arrays (what RobotTaskEnv.compute_reward, core.py:226, is called with by a CPU learner). */
int pg_compute_reward_host(int task, int reward_type, double threshold, const void* achieved_goal, const void* desired_goal,
                           float* reward, long long m, int dtype, int device);
int pg_is_success_host(int task, double threshold, const void* achieved_goal, const void* desired_goal, unsigned char* success,
                       long long m, int dtype, int device);
/* The two _host calls above stage through per-device buffers that only grow: number of (re)allocations so far (diagnostic). */
long long pg_host_stage_allocations(void);

/* RobotTaskEnv.save_state / restore_state / remove_state (core.py:252-278; pybullet.py:61-68,266-280): bit-exact device
 * snapshot of the whole batch (state, goals, episode counters).  Save and restore are one device-to-device copy enqueued on
 * `stream`, with no synchronisation: with NULL (the legacy default stream), synchronise it if you need the copy complete.  A removed
 * snapshot's buffer is reused by the next save, so a save / restore / remove loop allocates nothing after its first round and can be
 * captured in a CUDA graph. */
int pg_save_state(pg_env* env, int* state_id, void* stream);
int pg_restore_state(pg_env* env, int state_id, void* stream);
int pg_remove_state(pg_env* env, int state_id);

/* Raw state exchange for the facade getters/setters (pybullet.py:284-460) and the parity tests: float64 rows
 * [q(9) qd(9) | per object: pos(3) quat(4) lin(3) ang(3) | goal(G) | episode step], state_dim wide. */
int pg_get_state(pg_env* env, double* state, void* stream);
int pg_set_state(pg_env* env, const double* state, const unsigned char* mask, void* stream);
/* calculateInverseKinematics on link 11 from the current joint state (pybullet.py:479-497): target [N,3] + quat [N,4]
 * float64 -> joint angles [N,7] float64. */
int pg_inverse_kinematics(pg_env* env, const double* position, const double* orientation, double* joint_angles, void* stream);
/* The same call for any link 0..11 (PyBullet.inverse_kinematics(body, link, ...), pybullet.py:479-497; the reference's known-answer
 * test uses link 6, test/pybullet_test.py:254-266): all nine joint values per row, [N,9] float64. */
int pg_inverse_kinematics_link(pg_env* env, int link, const double* position, const double* orientation, double* joint_angles, void* stream);
/* getLinkState of any link 0..11 (PyBullet.get_link_position / _orientation / _velocity / _angular_velocity, pybullet.py:351-400):
 * rows [pos3 quat4 (x,y,z,w) lin3 ang3] float64 of the link's CoM frame; like pybullet without computeForwardKinematics, the pose
 * comes from the link-transform cache (one sub-step stale) and the velocity is rotated by the cached basis. */
int pg_get_link_state(pg_env* env, int link, double* out, void* stream);

/* End-effector (link 11) pose from the current joint state, rows [x y z qx qy qz qw] float64 (the fork's get_ee_position /
 * get_ee_orientation, panda_gym/envs/robots/panda_cartesian.py:218-225). */
int pg_get_ee_pose(pg_env* env, double* pose, void* stream);

/* The fork's scripted motion primitives (panda_gym/envs/robots/panda_cartesian.py:47-68: move, grasp, release) for every env of an
 * ee-controlled task handle.  A pg_motion plan is bound to a batch size and a device and serves any handle of that size on that
 * device.  Each env runs its own primitive with its own step count; a primitive begun on an env replaces the one it was running.
 *   move: way-points 1.5 cm apart (20 for a distance under 3 cm) from the EE position when the move begins to goal_pos [N,3], and a
 *     Slerp from the EE orientation then to goal_quat [N,4] (x,y,z,w; float64, normalised inside).  Each step's action is the next
 *     way-point minus the current EE position, finger action 0.
 *   gripper: `steps` steps of zero displacement with the finger action finger_action (grasp: -1, 30 steps; release: width, 30 steps),
 *     holding the current EE orientation.  Not for the blocked-gripper tasks Reach, Push and Slide (PG_ERR_STATE).
 * mask [N] (DEVICE, NULL = all) selects the envs a primitive begins on.  pg_motion_step writes each env's action and target
 * orientation (an env with no primitive left gets zero displacement, finger action 0 and its current orientation), then runs
 * pg_step with the plan's orientations on `stream` without auto-reset, and writes remaining [N] (int32, may be NULL): the steps of the env's primitive
 * still to take.  The primitives use the fork's unscaled actions: set pg_set_action_scale(env, 1.0, 1.0).  Plan state is not part
 * of pg_save_state snapshots.  Errors: NULL plan or env, or a plan of another size or device, PG_ERR_ARG; a bare or joint-controlled
 * handle PG_ERR_STATE; steps < 0 PG_ERR_ARG. */
typedef struct pg_motion pg_motion;
int pg_motion_create(int num_envs, int device, pg_motion** out);
int pg_motion_destroy(pg_motion* plan);
int pg_motion_move(pg_motion* plan, pg_env* env, const double* goal_pos, const double* goal_quat, const unsigned char* mask, void* stream);
int pg_motion_gripper(pg_motion* plan, pg_env* env, double finger_action, int steps, const unsigned char* mask, void* stream);
int pg_motion_step(pg_motion* plan, pg_env* env, float* obs, float* achieved_goal, float* desired_goal, float* reward,
                   unsigned char* terminated, unsigned char* truncated, int* remaining, void* stream);

/* The fork's camera path, PyBullet.render (panda_gym/pybullet.py:149-264) with the camera of get_cam2world_transforms (:70-107), for
 * every env of the handle: camera = {target x, y, z, distance, yaw, pitch, roll} (HOST, degrees; the reference's defaults are
 * {0,0,0, 1.4, 45, -30, 0}), fov 60, near 0.1, far 100.  Analytic ray casting of the primitives the kernels simulate (plane, table,
 * free bodies, the robot as its physics boxes -- its visual meshes are not in the reference tree).  DEVICE outputs, each may be NULL:
 * depth [N,H,W] float32 = OpenGL depth-buffer values as getCameraImage returns them (1.0 = nothing hit); rgba [N,H,W,4] uint8 (flat
 * body colours of the task scenes, diffuse shading); segmentation [N,H,W] uint8 (0 background, 1 plane, 2 table, 3/4 objects,
 * 5 robot base, 6 + link); points [N,H,W,3] float32 = the reference's deprojection of every pixel through inv(P V) (NaN where
 * filtered) with valid [N,H,W] uint8: depth buffer < 0.99 and, with crop != 0, the workspace box 0 < z < 0.67, -0.5 < x < 0.2. */
int pg_render(pg_env* env, int width, int height, const double* camera, int crop, float* depth, unsigned char* rgba,
              unsigned char* segmentation, float* points, unsigned char* valid, void* stream);

/* Episode statistics accumulated by auto-reset since creation: {episodes, successes, return_sum, length_sum} (host). */
int pg_stats(pg_env* env, double out[4]);
/* Number of env-steps that ended in a non-finite state (counted; with auto_reset the env is truncated and restarted). */
int pg_diverged(pg_env* env, long long* count);
/* Number of contact candidates dropped because an env already held the per-sub-step cap (10 contacts for scenes with at most one
 * object, 22 for Stack -- the size of the on-chip contact store; PyBullet has no such cap, the oracle applies the same one). */
int pg_contact_overflows(pg_env* env, long long* count);
/* Scheduling introspection (host buffers): the per-env 16-bit key written by the last launch and the thread -> env map built from
 * the previous one (bits 0-4 contacts at the end of the launch, bit 5 robot contact, bit 6 solver ran all sweeps, bit 7 near a
 * contact, bit 9 full joint-limit sweep, bits 10-13 generic contacts (Stack)). */
int pg_debug_schedule(pg_env* env, unsigned short* key, int* perm);
/* Timing introspection (handles created with PG_DEBUG_TIMING=1 in the environment): per thread slot of the last launch, the SM
 * cycles spent in the env's step code and the key it wrote; out is a host buffer of num_envs x 2 int64. */
int pg_debug_timing(pg_env* env, long long* out);
/* Number of kernels this library has launched in this process. */
long long pg_kernel_launches(void);
const char* pg_last_error(void);

#ifdef __cplusplus
}
#endif
#endif
