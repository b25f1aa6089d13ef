/*
 * salp_b200.h -- C ABI of the B200-native batched SALP simulator.
 *
 * This is the drop-in boundary for ONE hot path of Avielstein/GRASP_LAB_SALP:
 * SalpRobotEnv.reset()/step() and everything under it (robot.py, dynamics.py,
 * geometry.py), batched over N independent environments on one GPU.
 *
 * The reference is pure Python and has no FFI; the "interface each entry point
 * replaces" is therefore a Python method of the reference (file:line given at
 * each declaration, paths relative to the reference's src/).  INTEGRATION.md
 * shows the ctypes stub a maintainer adds to bind it.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types cross this boundary;
 *   - every function returns 0 (SALP_OK) or a negative SalpStatus; nothing
 *     throws; salp_last_error() gives the message of the last failure;
 *   - "_dev" pointers are device pointers on the handle's GPU, owned by the
 *     caller; "_host" pointers are host memory (pinned memory makes the copies
 *     asynchronous but is not required);
 *   - all device work is enqueued on the caller's stream (cudaStream_t passed
 *     as void*; NULL = legacy default stream); no hidden synchronisation in the
 *     *_dev entry points; the *_host entry points synchronise the stream before
 *     they return;
 *   - a handle is not re-entrant (one call in flight); distinct handles (one
 *     per GPU / rank) are independent.
 */
#ifndef SALP_B200_H
#define SALP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SALP_ABI_VERSION 1
#define SALP_MAX_OBSTACLES 8
#define SALP_OBS_BASE 6            /* salp_robot_env.py:658-665 */
#define SALP_NUM_REWARD_TERMS 8    /* 7 components (salp_robot_env.py:387-395) + total */
#define SALP_NUM_EPISODE_METRICS 20

typedef enum SalpStatus {
  SALP_OK = 0,
  SALP_ERR_INVALID = -1,      /* bad argument */
  SALP_ERR_CUDA = -2,         /* CUDA runtime failure (message in salp_last_error) */
  SALP_ERR_NO_DEVICE = -3,    /* no usable sm_100 GPU: there is NO CPU fallback */
  SALP_ERR_RANGE = -4,        /* an action drove the cycle past SALP_MAX_SUBSTEPS */
  SALP_ERR_ALLOC = -5,
  SALP_ERR_HANDOFF = -6       /* SALP_STEP_CHECK_HANDOFF: a pipeline-kernel warp read a ring row that was not the one written for it */
} SalpStatus;

/* Arithmetic the substep loop runs in. */
typedef enum SalpPrecision {
  SALP_PRECISION_F64 = 0,     /* quirk-for-quirk float64 restatement ("reference mode") */
  SALP_PRECISION_MIXED = 1    /* fp32 motion state, fp64 finite-difference core + accumulators */
} SalpPrecision;

/* SalpParams.randomization: the reference's default-off robustness switches, sampled on the device
 * from counter-based Philox streams keyed by (seed, global env id, episode, cycle): statistical,
 * not bitwise, parity with the reference's global np.random draws.  SALP_PRECISION_MIXED only. */
#define SALP_RAND_ACTION 1u        /* SalpRobotEnv.enable_action_randomization, salp_robot_env.py:176-181: +-10 % */
#define SALP_RAND_OBSERVATION 2u   /* enable_observation_randomization, :183-194 */
#define SALP_RAND_DYNAMICS 4u      /* Robot.enable_dynamic_randomization, robot.py:594-628: 7 coefficient groups +-50 % per cycle */
#define SALP_RAND_DISTURBANCE 8u   /* Robot.enable_disturbances, robot.py:210-242, 796-838: OU force (x, y) / torque (z) noise */
#define SALP_RAND_LATENCY 16u      /* enable_latency, salp_robot_env.py:294-297: the extra set_control (cycle += 1) */

/* salp_step flags */
#define SALP_STEP_AUTORESET 1u     /* SB3 VecEnv semantics: reset finished envs, obs = post-reset obs */
#define SALP_STEP_SORT_BY_K 2u     /* balance warps: order envs by substep count before the loop */
/* Kernel choice for small batches (N <= 64 envs per SM, MIXED).  Default there: the warp-specialised
 * pipeline kernel (shape / coefficient / dynamics / kinematics warps); results are bit-identical
 * with the fused one-warp kernel. */
#define SALP_STEP_PIPELINE 4u      /* accepted for compatibility: the pipeline kernel is the default where it applies */
#define SALP_STEP_FUSED 8u         /* force the fused one-warp kernel */
/* The loop has a form for axisymmetric coefficient sets (axes 1 and 2 alike, as in the defaults) that
 * shares their entries; it is chosen automatically and gives the same bits as the general form. */
#define SALP_STEP_GENERIC 16u      /* force the general form (tests) */
/* Checked hand-off (tests): the pipeline kernel tags every shared-memory ring row with the substep it
 * was written for and verifies the tag on the consuming warp; a mismatch sets SALP_ERR_HANDOFF in the
 * sticky status (salp_check).  Same results, a few per cent slower. */
#define SALP_STEP_CHECK_HANDOFF 32u

/*
 * Every literal the reference hard-codes on this path, as one POD.
 * salp_default_params() fills it with the values below.
 */
typedef struct SalpParams {
  /* Nozzle(...)  train_robot.py:13, robot.py:20-44 */
  double nozzle_length1, nozzle_length2, nozzle_length3;
  double nozzle_area, nozzle_mass;
  double nozzle_gamma;          /* robot.py:42  pi/4 */
  double nozzle_angle_speed;    /* robot.py:43  31*pi/30 */
  /* Robot(...)  train_robot.py:14-17, robot.py:285-295 */
  double dry_mass, init_length, init_width, max_contraction;
  double density;               /* set_environment(1000), train_robot.py:17 */
  double dt;                    /* robot.py:293 */
  double buoy_mass, skin_mass, tube_mass, tube_volume;
  /* coefficient means, robot.py:300-306 (diagonals) */
  double discharge_coefficient, drag_force_ratio, drag_torque_ratio;
  double added_mass_force[3], added_mass_rate_force[3];
  double added_mass_torque[3], added_mass_rate_torque[3];
  /* robot.py:415-434: rows x,y,z; columns [initial, fully contracted] */
  double trans_drag_range[6], rot_drag_range[6];
  /* np.polyfit(deg 2) of geometry.py:6-10 and :17-21, highest power first */
  double refill_poly[3], jet_poly[3];
  /* SalpRobotEnv(...) salp_robot_env.py:35-47, 471-482 */
  double tank_x_min, tank_x_max, tank_y_min, tank_y_max;
  double target_radius, obstacle_radius;
  double out_of_bounds_distance;      /* salp_robot_env.py:265 */
  double success_bonus, out_of_bounds_penalty, collision_penalty, timeout_penalty;
  int32_t max_cycles;                 /* salp_robot_env.py:274 */
  int32_t num_obstacles;              /* <= SALP_MAX_OBSTACLES */
  int32_t precision;                  /* SalpPrecision */
  int32_t randomization;              /* SALP_RAND_* bits; 0 = the reference's defaults (everything off) */
} SalpParams;

typedef struct SalpSim* salp_handle;

/* Buffers of one salp_step call.  N = num_envs, D = SALP_OBS_BASE + 2*num_obstacles. */
typedef struct SalpStepIO {
  const float* actions;       /* in  [N,3]  raw Box actions (salp_robot_env.py:63-67), NOT clipped */
  float* obs;                 /* out [N,D]  _get_observation(); post-reset obs where auto-reset fired */
  float* reward;              /* out [N]    */
  uint8_t* terminated;        /* out [N]    `done`      salp_robot_env.py:262-264 */
  uint8_t* truncated;         /* out [N]    `truncated` salp_robot_env.py:265-276 */
  float* terminal_obs;        /* out [N,D]  nullable: obs of the finished episode (== obs if not reset) */
  double* reward_terms;       /* out [N,8]  nullable: track,heading,smooth,yaw,time,sideslip,obstacle,total(f64, with terminal bonuses) */
  int32_t* substeps;          /* out [N]    nullable: K = physics substeps run this cycle */
  double* episode_metrics;    /* out [N,SALP_NUM_EPISODE_METRICS] nullable; row valid where terminated|truncated */
} SalpStepIO;

/* Row layout of SalpStepIO.episode_metrics (salp_robot_env.py:399-447 + SB3 Monitor r/l) */
typedef enum SalpEpisodeMetric {
  SALP_EM_RETURN = 0,           /* Monitor info["episode"]["r"] */
  SALP_EM_LENGTH = 1,           /* Monitor info["episode"]["l"] */
  SALP_EM_PATH_LENGTH = 2,
  SALP_EM_DIRECT_DISTANCE = 3,
  SALP_EM_PATH_EFFICIENCY = 4,
  SALP_EM_FINAL_DISTANCE = 5,
  SALP_EM_INITIAL_DISTANCE = 6,
  SALP_EM_AVG_COMPRESSION = 7,
  SALP_EM_AVG_COAST_TIME = 8,
  SALP_EM_AVG_NOZZLE_ANGLE = 9,
  SALP_EM_AVG_VELOCITY = 10,
  SALP_EM_AVG_REWARD_TRACK = 11,  /* ..17: avg_rewards_{track,heading,smooth,yaw,time,sideslip,obstacle} */
  SALP_EM_TOTAL_SUBSTEPS = 18,
  SALP_EM_NONFINITE = 19        /* 1.0 if the episode was cut because the state became non-finite (see salp_step) */
} SalpEpisodeMetric;

/*
 * Per-env state columns readable / writable through salp_get_state / salp_set_state
 * (used by the parity tests to inject and compare state; names follow robot.py).
 * All F64 fields are double, F32 float, I32 int32_t, one value per env.
 */
typedef enum SalpField {
  /* F64: Robot motion state, robot.py:358-374 */
  SALP_F_VEL_X = 0, SALP_F_VEL_Y, SALP_F_VEL_Z,                 /* velocity (body frame) */
  SALP_F_ANGVEL_X, SALP_F_ANGVEL_Y, SALP_F_ANGVEL_Z,            /* angular_velocity */
  SALP_F_EULER_X, SALP_F_EULER_Y, SALP_F_EULER_Z,               /* euler_angle */
  SALP_F_POSW_X, SALP_F_POSW_Y, SALP_F_POSW_Z,                  /* position_world */
  SALP_F_ACC_X, SALP_F_ACC_Y, SALP_F_ACC_Z,                     /* acceleration (of the last substep) */
  SALP_F_ANGACC_X, SALP_F_ANGACC_Y, SALP_F_ANGACC_Z,            /* angular_acceleration */
  SALP_F_POS_X, SALP_F_POS_Y, SALP_F_POS_Z,                     /* position (body-frame integral) */
  SALP_F_ANGLE_X, SALP_F_ANGLE_Y, SALP_F_ANGLE_Z,               /* angle */
  SALP_F_PREVPOS_X, SALP_F_PREVPOS_Y, SALP_F_PREVPOS_Z,         /* prev_position */
  SALP_F_PREVANGLE_X, SALP_F_PREVANGLE_Y, SALP_F_PREVANGLE_Z,   /* prev_angle */
  /* F64: geometry tail, robot.py:325-339 */
  SALP_F_LENGTH, SALP_F_WIDTH, SALP_F_PREV_VOLUME,
  SALP_F_PREV_I_X, SALP_F_PREV_I_Y, SALP_F_PREV_I_Z,
  SALP_F_COM_X, SALP_F_PREV_COM_X, SALP_F_COM_RATE_X, SALP_F_PREV_COM_RATE_X, SALP_F_COM_ACC_X,
  /* F64: nozzle, robot.py:31-44 */
  SALP_F_NOZZLE_ANGLE1, SALP_F_NOZZLE_ANGLE2,
  /* F64: env, salp_robot_env.py:127,146-153 */
  SALP_F_PREV_DIST, SALP_F_SPEED_WORLD,
  SALP_F_EP_RETURN, SALP_F_EP_PATH_LENGTH, SALP_F_EP_INITIAL_DISTANCE,
  SALP_F_EP_SUM_A0, SALP_F_EP_SUM_A1, SALP_F_EP_SUM_ABS_A2, SALP_F_EP_SUM_SPEED,
  SALP_F_EP_SUM_TERM0, SALP_F_EP_SUM_TERM1, SALP_F_EP_SUM_TERM2, SALP_F_EP_SUM_TERM3,
  SALP_F_EP_SUM_TERM4, SALP_F_EP_SUM_TERM5, SALP_F_EP_SUM_TERM6,
  SALP_F_EP_SUBSTEPS,
  SALP_F_OU_FORCE_X, SALP_F_OU_FORCE_Y, SALP_F_OU_TORQUE_Z,     /* OUDisturbance.state (robot.py:279-280), SALP_RAND_DISTURBANCE */
  SALP_NUM_F64_FIELDS,

  /* F32 columns */
  SALP_F32_BASE = 1000,
  SALP_F_NOZZLE_YAW = SALP_F32_BASE,                            /* nozzle.yaw (np.float32) */
  SALP_F_PREV_ACTION0, SALP_F_PREV_ACTION1, SALP_F_PREV_ACTION2,
  SALP_F_TARGET_X, SALP_F_TARGET_Y,
  SALP_F_OBSTACLE0_X,                                           /* + 2*i (+1 for y), i < SALP_MAX_OBSTACLES */
  SALP_F32_END = SALP_F_OBSTACLE0_X + 2 * SALP_MAX_OBSTACLES,

  /* I32 columns */
  SALP_I32_BASE = 2000,
  SALP_F_PHASE = SALP_I32_BASE,                                 /* Robot.state.value: 0 REFILL 1 JET 2 COAST 3 REST */
  SALP_F_CYCLE,                                                 /* Robot.cycle */
  SALP_F_EP_LENGTH,                                             /* env steps in the running episode */
  SALP_F_EPISODE_INDEX,                                         /* episodes started by this env (reset counter) */
  SALP_I32_END
} SalpField;

/* ---- construction ------------------------------------------------------------------- */

/* Literals of make_env() (train_robot.py:11-21), Robot.__init__ (robot.py:261-308) and
 * SalpRobotEnv.__init__ (salp_robot_env.py:35-47).  The two timing polynomials are fitted
 * here by least squares on the reference's data points (geometry.py:6-10, 17-21); a Python
 * host overwrites them with np.polyfit's own bits. */
int salp_default_params(SalpParams* out);

/* Replaces: make_vec_env(make_env, n_envs) (train_robot.py:26) -- N x { Nozzle, Robot,
 * SalpRobotEnv.__init__ }.  `env_id_offset` is the global index of env 0 (multi-GPU shards
 * pass rank * N so per-env random streams do not depend on the sharding). */
int salp_create(const SalpParams* params, int64_t num_envs, int device, uint64_t seed,
                int64_t env_id_offset, salp_handle* out);
int salp_destroy(salp_handle h);

int64_t salp_num_envs(salp_handle h);
int32_t salp_obs_dim(salp_handle h);
const char* salp_last_error(salp_handle h);   /* h may be NULL: error of the last failed salp_create */
const char* salp_build_info(void);            /* "sm_100a nvcc 12.9 ..." */

/* ---- the hot path ------------------------------------------------------------------- */

/* Replaces: SalpRobotEnv.reset() (salp_robot_env.py:114-155) incl. Robot.reset()
 * (robot.py:452-501), generate_target_point("random") (:449-533), _generate_obstacles
 * (:535-559).  mask_dev: uint8[N], nullable = reset every env.  obs_dev: float[N,D] nullable. */
int salp_reset(salp_handle h, const uint8_t* mask_dev, float* obs_dev, void* stream);

/* Replaces: SalpRobotEnv.step() (salp_robot_env.py:196-299) incl. Nozzle.set_yaw_angle /
 * solve_angles (robot.py:62-98), Robot.set_control (:544-592), Robot.step_through_cycle
 * (:740-776) and the K x Robot.step() substep loop (:670-678) with every dynamics.py /
 * geometry.py function under it; plus, with SALP_STEP_AUTORESET, the auto-reset that SB3's
 * DummyVecEnv/SubprocVecEnv worker performs around it.
 *
 * Where the reference raises: some contractions (a0 in about [0.0905, 0.094], jet_time a
 * fraction of one substep) make the reference's integrator diverge; its state overflows and
 * np.linalg.solve (dynamics.py:6-10) throws LinAlgError, i.e. the reference process dies.  A
 * batched call cannot raise per env: such an env is TRUNCATED in the step whose cycle left its
 * state non-finite (truncated = 1, terminated = 0, reward = -out_of_bounds_penalty, observation
 * with non-finite entries replaced by 0, episode metric SALP_EM_NONFINITE = 1). */
int salp_step(salp_handle h, const SalpStepIO* io_dev, uint32_t flags, void* stream);

/* Same two calls with HOST buffers; they return when the results are in the caller's memory
 * (one stream synchronise).  This is what a numpy-facing VecEnv calls.  Any host memory works.
 * Transport of salp_step_host: for PAGE-LOCKED buffers (cudaHostAlloc / cudaHostRegister, e.g.
 * torch's pin_memory) in SALP_PRECISION_MIXED without SALP_STEP_SORT_BY_K the kernel writes obs,
 * reward, flags and terminal obs directly into the caller's memory while it runs (and reads the
 * actions in place for N <= 18944); otherwise H2D of the actions, the kernels on internal device
 * buffers, one D2H per non-null output.  Results are bit-identical either way. */
int salp_reset_host(salp_handle h, const uint8_t* mask_host, float* obs_host);
int salp_step_host(salp_handle h, const SalpStepIO* io_host, uint32_t flags);

/* ---- parity / tooling --------------------------------------------------------------- */

/* Scene pool: replaces the reference's *global np.random* draws in reset() by caller-given
 * scenes so that an external oracle can be driven with identical targets/obstacles.
 * targets_host: float[N,P,2]; obstacles_host: float[N,P,num_obstacles,2]; episode e of env i
 * uses scene (e mod P).  P = 0 returns to the built-in Philox sampler. */
int salp_set_scene_pool(salp_handle h, const float* targets_host, const float* obstacles_host,
                        int64_t scenes_per_env);

/* Copy one state field of `count` envs from `first` to / from a DENSE host array (synchronous). */
int salp_get_state(salp_handle h, int32_t field, void* host_dst, int64_t first, int64_t count);
int salp_set_state(salp_handle h, int32_t field, const void* host_src, int64_t first, int64_t count);
/* Raw device address of env 0's element of a field and the byte stride between consecutive envs
 * (state is stored as one record per env): zero-copy strided views for torch / cupy. */
int salp_state_ptr(salp_handle h, int32_t field, void** dev_ptr, int64_t* stride_bytes);

/* History feed -- replaces Robot.enable_history_recording() + the per-substep histories of
 * Robot.step_through_cycle (robot.py:681-776) that SalpRobotEnv.step hands out as
 * info["position_history" | "length_history" | "width_history"] (salp_robot_env.py:279-284) and the
 * viewer / plotting tools read.  Runs the NEXT cycle of ONE env for `action_host[3]` in float64
 * reference arithmetic on a scratch copy of its state (the env is NOT advanced) and writes one row
 * per substep, taken after Robot.step() like the reference's histories:
 *   row = [position_world xyz, euler_angle xyz, velocity xyz, angular_velocity xyz, length, width]
 * trace_host: double[capacity][SALP_TRACE_WIDTH]; *substeps_out = K (rows beyond capacity are dropped). */
#define SALP_TRACE_WIDTH 14
int salp_trace_cycle(salp_handle h, int64_t env, const float* action_host, double* trace_host, int32_t capacity,
                     int32_t* substeps_out);

/* Sticky device-side status (e.g. SALP_ERR_RANGE); reading it synchronises the device. */
int salp_check(salp_handle h);

/* Kernel launches issued by this handle so far (bench.py reports it as gpu_launches). */
int64_t salp_launch_count(salp_handle h);
/* Name of the step kernel the last salp_step / salp_step_host call launched (the launcher picks by
 * batch size, precision and flags); static string, "" before the first step. */
const char* salp_last_step_kernel(salp_handle h);

/* Layout checks for bindings that mirror the structs (ctypes): a host whose mirror disagrees with
 * these must refuse to drive the library. */
int32_t salp_abi_version(void);
int64_t salp_sizeof_params(void);
int64_t salp_sizeof_step_io(void);

/* Measurement tooling (no reference counterpart): register-resident FFMA micro-benchmark on
 * `device`; writes the sustained FP32 rate in TFLOP/s (2 flop per FMA) over ~`millis` ms.
 * bench.py uses it as the denominator of the FP32-pipe roofline (MEASURED_PEAKS.json has no
 * FP32 SIMT figure). */
int salp_probe_fp32_peak(int device, int millis, double* tflops_out);

/* Diagnostic: salp_step with flag bit 29 (0x20000000) makes block 0 of the small-batch pipeline kernel
 * record clock64() at the boundaries of its prologue, substep loops and epilogue; this reads the 16
 * words back (tools/diag_stamps.py explains them).  Synchronises the device. */
int salp_debug_p4_stamps(long long* out16);

/* ---- rollout-side policy forward (no reference counterpart in src/: the reference's policies live in
 * stable-baselines3; this is SB3's `MlpPolicy` forward as one kernel in front of salp_step) ----------
 * weights_dev: one packed float array -- actor W1[64,D] b1[64] W2[64,64] b2[64] W3[3,64] b3[3], critic
 * W1[64,D] b1[64] W2[64,64] b2[64] W3[1,64] b3[1], log_std[3] (row-major like torch's nn.Linear.weight);
 * salp_mlp_packed_size(D) floats.  noise_dev: standard-normal [N,3].  Outputs: action [N,3] = mean +
 * noise * exp(log_std), clipped [N,3] = action clipped to [low, high] (what the env gets), logp [N], value [N].
 * action_low / action_high: host float[3].
 * Deterministic mode (SB3 predict(deterministic=True)): noise_dev NULL gives action = mean exactly, clipped =
 * the mean clipped to [low, high]; logp_dev may then be NULL (not written).  value_dev NULL skips the critic.
 * With noise_dev given, logp_dev and value_dev are mandatory. */
int64_t salp_mlp_packed_size(int32_t obs_dim);
int salp_mlp_act(const float* weights_dev, int32_t obs_dim, const float* obs_dev, const float* noise_dev, int64_t n,
                 const float* action_low, const float* action_high, float* action_dev, float* clipped_dev,
                 float* logp_dev, float* value_dev, void* stream);

/* ---- rollout-side LSTM cell on the tensor cores (sb3_contrib RecurrentPPO's MlpLstmPolicy as the
 * reference configures it, src/train_robot_recurrent_ppo.py:100-105: lstm_hidden_size = 256, separate
 * actor / critic LSTMs on the flattened observation; the episode-start state reset is sb3_contrib's
 * _process_sequence).  One step of torch.nn.LSTMCell(obs_dim, 256) for N envs:
 *     gates = obs W_ih^T + (h keep) W_hh^T + b_ih + b_hh      keep[e] = starts[e] ? 0 : 1
 *     i, f, o = sigmoid; g = tanh; c' = f (c keep) + i g; h' = o tanh(c')        (gate order i, f, g, o)
 * as a bf16 x bf16 -> fp32 tcgen05 GEMM (TMA operands, TMEM accumulator) with the cell update fused
 * behind it (csrc/salp_lstm.cu).  hidden must be 256, obs_dim <= 64.
 * salp_lstm_pack_weights: once per set of weights -- permutes / rounds [W_hh | W_ih] into
 *   packed_dev (salp_lstm_weight_bytes() bytes) and b_ih + b_hh into bias_dev (float[1024]).
 * salp_lstm_cell: h / c [N, 256] fp32, in place allowed (h_out == h_in, c_out == c_in); starts_dev: N
 *   bytes (torch.bool) or NULL; scratch_dev: salp_lstm_scratch_bytes(N) bytes, 16-byte aligned.
 * salp_lstm_check: synchronises; SALP_ERR_CUDA if a kernel gave up waiting on one of its barriers. */
int64_t salp_lstm_weight_bytes(void);
int64_t salp_lstm_scratch_bytes(int64_t n);
int salp_lstm_pack_weights(const float* w_ih_dev, const float* w_hh_dev, const float* b_ih_dev, const float* b_hh_dev,
                           int32_t obs_dim, int32_t hidden, void* packed_dev, float* bias_dev, void* stream);
int salp_lstm_cell(const void* packed_dev, const float* bias_dev, const float* obs_dev, const uint8_t* starts_dev,
                   const float* h_in_dev, const float* c_in_dev, float* h_out_dev, float* c_out_dev, void* scratch_dev,
                   int64_t n, int32_t obs_dim, int32_t hidden, void* stream);
int salp_lstm_check(void);

/* ---- rollout-side SAC actor (stable-baselines3 SACPolicy as src/train_robot.py trains it: actor
 * net_arch [256, 256], ReLU, squashed Gaussian; csrc/salp_sac.cu).  For N envs in one launch:
 *     latent = ReLU(W2 ReLU(W1 obs + b1) + b2);  mu = Wmu latent + bmu;
 *     log_std = clamp(Wls latent + bls, -20, 2);  u = mu + exp(log_std) noise  (noise_dev NULL: u = mu);
 *     scaled = tanh(u) (what the replay stores);  env = low + (scaled + 1) / 2 (high - low) (what salp_step gets)
 * Hidden size 256 and act_dim 3 are fixed; 1 <= obs_dim <= 64.  Layer 1 and the heads are fp32 (layer 1 an
 * fmaf chain over the inputs in order, from b1); layer 2 runs on the tensor cores (tcgen05) with bf16 operands
 * and fp32 accumulation.  Weights are torch nn.Linear layouts ([out, in], row-major, fp32, device memory).
 * salp_sac_weight_bytes: size of packed_dev (< 0 for an invalid obs_dim).
 * salp_sac_pack_weights: once per weight update; packed_dev 16-byte aligned.
 * salp_sac_act: obs [N, obs_dim], noise [N, 3] standard normal or NULL, outputs [N, 3]; action_low / high:
 *   host float[3].  Runs on the device that owns packed_dev.
 * salp_sac_check: synchronises the current device; SALP_ERR_CUDA if a kernel gave up on a bounded barrier wait.
 * Grouped (K = num_agents actors of one population in one launch, 1 <= K <= 65535): the parameters are stacked
 *   [K, ...] with the per-agent layout above; packed_dev holds K images of salp_sac_weight_bytes(obs_dim) bytes,
 *   image k byte-identical to what salp_sac_pack_weights writes for agent k (one launch packs all K).  Rows
 *   [k n, (k + 1) n) of obs, noise and the outputs belong to agent k (n = envs_per_agent >= 1), and agent k's rows
 *   are bit-identical to salp_sac_act on image k and those rows.  salp_sac_act / salp_sac_pack_weights are K = 1. */
int64_t salp_sac_weight_bytes(int32_t obs_dim);
int salp_sac_pack_weights(const float* w1, const float* b1, const float* w2, const float* b2,
                          const float* w_mu, const float* b_mu, const float* w_log_std, const float* b_log_std,
                          int32_t obs_dim, void* packed_dev, void* stream);
int salp_sac_act(const void* packed_dev, int32_t obs_dim, const float* obs_dev, const float* noise_dev,
                 int64_t n, const float* action_low, const float* action_high,
                 float* env_action_dev, float* scaled_action_dev, void* stream);
int salp_sac_pack_weights_grouped(const float* w1, const float* b1, const float* w2, const float* b2,
                                  const float* w_mu, const float* b_mu, const float* w_log_std, const float* b_log_std,
                                  int32_t num_agents, int32_t obs_dim, void* packed_dev, void* stream);
int salp_sac_act_grouped(const void* packed_dev, int32_t num_agents, int32_t obs_dim, const float* obs_dev,
                         const float* noise_dev, int64_t envs_per_agent, const float* action_low,
                         const float* action_high, float* env_action_dev, float* scaled_action_dev, void* stream);
int salp_sac_check(void);

/* ---- the element-wise halves of the LEARNER's LSTM step (RecurrentPPO update, BPTT; fp32, any hidden
 * size; csrc/salp_lstm_train.cu, used by grasp_lab_salp_b200/lstm_seq.py's autograd.Function) -----------
 * forward : gates [B, 4H] (torch order i, f, g, o; biases and both products already summed) ->
 *   act [B, 4H] = (sigmoid i, sigmoid f, tanh g, sigmoid o), c_out = f (c_prev keep_cur) + i g,
 *   h_out = o tanh(c_out), hm_next = h_out keep_next (the next step's GEMM operand; may be NULL).
 *   keep_* : float [B] (1 - episode_start) or NULL (= 1).
 * backward: dh = dh_ext + dh_rec keep_next (either may be NULL), dc_next (NULL = 0), the forward's act /
 *   c_cur (= its c_out) / c_prev / keep_cur -> dgates [B, 4H], dc_prev = dc f keep_cur. */
int salp_lstm_pointwise_fwd(const float* gates_dev, const float* c_prev_dev, const float* keep_cur_dev,
                            const float* keep_next_dev, int64_t batch, int32_t hidden, float* act_dev, float* c_out_dev,
                            float* h_out_dev, float* hm_next_dev, void* stream);
int salp_lstm_pointwise_bwd(const float* dh_ext_dev, const float* dh_rec_dev, const float* keep_next_dev,
                            const float* dc_next_dev, const float* act_dev, const float* c_cur_dev, const float* c_prev_dev,
                            const float* keep_cur_dev, int64_t batch, int32_t hidden, float* dgates_dev, float* dc_prev_dev,
                            void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SALP_B200_H */
