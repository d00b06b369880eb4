/* ssa_ukf.h — C ABI of libssa_ukf.so: the B200 (sm_100a) implementation of ssa-gym's per-step
 * estimation hot path (UKF predict/update over every resident space object of every environment).
 *
 * This is the drop-in boundary.  Everything above it (gym.Env reset/step, RNG, failure messages,
 * histories) stays Python; everything below is CUDA.  No torch types, only plain pointers/sizes.
 * Every entry point returns 0 on success or a negative SSA_E* code; nothing throws.  All calls on
 * one handle must come from one host thread; work is enqueued on the given CUDA stream and is
 * asynchronous unless the function name says download/sync.
 *
 * Reference interfaces replaced (file:line in the read-only upstream AshHarvey/ssa-gym):
 *   ssa_ukf_create        envs/ssa_tasker_simple_2.py:72-184  (__init__: dt, Q, R, observer, sigma-point
 *                         parameters; filterpy MerweScaledSigmaPoints weights) and :211-218 (UKF objects)
 *   ssa_ukf_reset         envs/ssa_tasker_simple_2.py:193-241 (reset: x_true[0], x_filter[0], P_0)
 *   ssa_ukf_predict       envs/ssa_tasker_simple_2.py:265-287 (truth fx loop + filters[j].predict())
 *                         -> filterpy UKF.predict -> envs/farnocchia.py:1053 fx, envs/dynamics.py:402 msqrt
 *   ssa_ukf_update        envs/ssa_tasker_simple_2.py:292-315 (hx, visibility gate, filters[a].update(z))
 *                         -> filterpy UKF.update -> envs/dynamics.py:219 hx, :342 mean_z, :260 residual_z
 *   ssa_ukf_step          the whole of step(): SS2:243-367, fused (truth + predict + update + obs/error)
 *   ssa_ukf_env_reduce    SS2:324-354 (reward / done), agents.py:7-9,35-42,66-81 (greedy taskers),
 *                         SS2:410-425 (visible_objects)
 *   ssa_ukf_scores        envs/reward.py:6-50
 *   ssa_ukf_download      the numpy arrays the reference env exposes: x_true, x_filter, P_filter, obs,
 *                         delta_pos, delta_vel, sigma_pos, sigma_vel, y, S, sigmas_h  (SS2:132-161)
 */
#ifndef SSA_UKF_H
#define SSA_UKF_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SSA_UKF_ABI_VERSION 1

/* error codes */
#define SSA_OK 0
#define SSA_EINVAL (-1)  /* bad argument */
#define SSA_ECUDA (-2)   /* CUDA runtime error; ssa_ukf_last_error() has the text */
#define SSA_ENOMEM (-3)
#define SSA_ENODEV (-4)  /* no CUDA device: there is no CPU fallback */

/* obs_type (SS2:100-107) */
#define SSA_OBS_AER 0
#define SSA_OBS_XYZ 1
/* reward_type (SS2:324-351) */
#define SSA_REWARD_JONES 0
#define SSA_REWARD_TRINARY 1
#define SSA_REWARD_SHAPED 2

/* Per-object status word (int32), also in ssa_gym_b200/csrc/ssa_ukf_core.h */
#define SSA_STATUS_FAILED 0x1
#define SSA_STATUS_LINALG 0x2
#define SSA_STATUS_NAN 0x4
#define SSA_STATUS_FXEXC 0x8
#define SSA_STATUS_TRUTHEXC 0x10
#define SSA_STATUS_IN_UPDATE 0x20

typedef struct ssa_ukf_cfg {
  int32_t abi_version;             /* SSA_UKF_ABI_VERSION */
  int32_t n_objects;               /* N = n_envs * m */
  int32_t n_envs;                  /* E; 1 for the drop-in env, N objects form E groups of m */
  int32_t m;                       /* rso_count: objects per environment */
  int32_t obs_type;                /* SSA_OBS_* */
  int32_t resample_after_predict;  /* 1: filterpy >= 1.4.5 predict() re-draws sigmas_f from the prior */
  int32_t reward_type;             /* SSA_REWARD_* (used by ssa_ukf_env_reduce) */
  int32_t n_steps;                 /* n: episode length (done when i+1 >= n) */
  double dt;                       /* time_step [s] */
  double lam_plus_n;               /* (lambda + n) of MerweScaledSigmaPoints */
  double Wm[13];                   /* mean weights, computed on the host with filterpy's expressions */
  double Wc[13];                   /* covariance weights */
  double Q[36];                    /* process noise, row-major 6x6 (Q_discrete_white_noise, SS2:110) */
  double R[9];                     /* measurement noise, row-major 3x3, added element-wise to S */
  double obs_itrs[3];              /* observer ECEF [m] (lla2ecef(obs_lla), SS2:94) */
  double T[9];                     /* trans_uvw_ecef(lat,lon), row-major (transformations.py:341-343) */
  double obs_limit;                /* elevation mask [rad] (SS2:85) */
} ssa_ukf_cfg;

typedef struct ssa_ukf ssa_ukf; /* opaque handle, owns all device buffers */

/* fields for ssa_ukf_download / ssa_ukf_upload / ssa_ukf_device_ptr.
 * Host layouts are the reference's numpy layouts (row-major):
 *   X_TRUE, X_FILTER  double[N][6]       P_FILTER double[N][6][6] (symmetric, mirrored from the packed upper)
 *   OBS               double[N][12] = [x(6), diag P(6)]  (results.py:60-72)
 *   DELTA_POS/VEL, SIGMA_POS/VEL, TRACE   double[N]      (results.py:36-47; np.trace)
 *   Z_TRUE, Y, Z_NOISE double[N][3]      S double[N][3][3]   SIGMAS_H double[N][13][3]
 *   VISIBLE uint8[N] (SS2:418-425)       STATUS int32[N]     INFLATIONS int32[N]
 *   ACTIONS int32[E]  REWARD double[E]  DONE uint8[E]  GREEDY int32[E][SSA_N_TASKERS]
 *   TRANS_ENV double[E][9] per-env trans_matrix  STEP_INDEX int32[E] per-env step counter i
 *   ENV_STATS double[E][4] = [max delta_pos, trinary reward, argmax sigma_pos, #visible]
 * Device layouts are struct-of-arrays with leading dimension ssa_ukf_ld(h) (see DESIGN.md).        */
enum ssa_field {
  SSA_F_X_TRUE = 0, SSA_F_X_FILTER = 1, SSA_F_P_FILTER = 2, SSA_F_OBS = 3,
  SSA_F_DELTA_POS = 4, SSA_F_DELTA_VEL = 5, SSA_F_SIGMA_POS = 6, SSA_F_SIGMA_VEL = 7, SSA_F_TRACE = 8,
  SSA_F_Z_TRUE = 9, SSA_F_Y = 10, SSA_F_S = 11, SSA_F_SIGMAS_H = 12, SSA_F_Z_NOISE = 13,
  SSA_F_VISIBLE = 14, SSA_F_STATUS = 15, SSA_F_INFLATIONS = 16,
  SSA_F_ACTIONS = 17, SSA_F_REWARD = 18, SSA_F_DONE = 19, SSA_F_GREEDY = 20, SSA_F_SCORES = 21,
  SSA_F_UPDATED = 22, SSA_F_TRANS_ENV = 23, SSA_F_STEP_INDEX = 24, SSA_F_ENV_STATS = 25,
  SSA_F_DIAG = 26,        /* double [N][2]: NEES, NIS (NaN where the object was not updated) - ssa_ukf_diagnostics */
  SSA_F_INNOV_FLAGS = 27, /* uint8 [N]: 0x80 valid | bit a: |y_a| < sqrt(S_aa) | bit 3+a: |y_a| < 2 sqrt(S_aa) */
  SSA_F_CATALOG_STATS = 28, /* double [5]: max delta_pos, sum of trinary counts, objects, max trace P, its index */
  SSA_F_ROLLOUT_OBS = 29,   /* device views of the episodic mode's output block: obs [N][12] ...              */
  SSA_F_ROLLOUT_REWARD = 30, /* ... and reward [E] (for an NCCL gather onto a learner's device)                 */
  SSA_F_ROLLOUT_ACTIONS = 31, /* int32 [E]: the device-side action buffer read by ssa_ukf_rollout_step(.., auto_reset | 2, ..) */
  SSA_F_ROLLOUT_DONE = 32,    /* uint8 [E]  and                                                                    */
  SSA_F_ROLLOUT_GREEDY = 33,  /* int32 [E][SSA_N_TASKERS] of the episodic output block                             */
  SSA_F_COUNT_
};

/* heuristic taskers evaluated on the device by ssa_ukf_env_reduce (agents.py) */
#define SSA_TASKER_NAIVE_GREEDY 0     /* argmax trace P over all objects           agents.py:7-9   */
#define SSA_TASKER_VISIBLE_GREEDY 1   /* argmax trace P over visible objects       agents.py:35-42 */
#define SSA_TASKER_POS_ERROR_GREEDY 2 /* argmax delta_pos over visible objects     agents.py:66-72 */
#define SSA_TASKER_VEL_ERROR_GREEDY 3 /* argmax delta_vel over visible objects     agents.py:75-81 */
#define SSA_TASKER_VISIBLE_GREEDY_AER 4 /* argmax of the 'aer' observation's trace column (nan/inf -> 0.001) over visible objects  agents.py:57-63 */
#define SSA_TASKER_SHANNON 5          /* argmax log(det P_i / det P_{i-1}) over visible objects   agents.py:15-26 */
#define SSA_N_TASKERS 6
/* a visible-* tasker returns -1 when the reference would fall back to action_space.sample()
 * (`not np.any(visible)` — also true when the only visible index is 0, agents.py:37).
 * SSA_TASKER_SHANNON keeps a determinant history per environment, keyed to the step index i the reduction runs at
 * (ssa_ukf_env_reduce's step_index or SSA_F_STEP_INDEX; the episodic mode's own counters): at a LARGER i than the
 * stored one the ratio is det P / det P of the stored step, which then becomes the history; at the SAME i it is
 * evaluated against the same previous determinant again and nothing moves, so repeated calls at one step give the
 * same picks; at i = 0, a smaller i, or with no history (after ssa_ukf_reset) the history restarts with ratio 1 and
 * the first visible object is picked.                                                                                */

/* flags for ssa_ukf_step */
#define SSA_STEP_TRUTH 0x1        /* propagate the true states (SS2:265-266) */
#define SSA_STEP_PREDICT 0x2      /* UKF predict on every non-failed object (SS2:271-287) */
#define SSA_STEP_UPDATE_ALL 0x4   /* catalog mode: update every object with its z_noise */
#define SSA_STEP_UPDATE_ACT 0x8   /* RL mode: update object actions[e] of each env e (SS2:292-315) */
#define SSA_STEP_EPILOGUE 0x10    /* obs / error / trace / visibility (SS2:320-322, 410-425) */
#define SSA_STEP_RECORD 0x20      /* also store z_true, y, S, sigmas_h of updated objects (SS2:298-304) */
#define SSA_STEP_M_PER_ENV 0x40   /* vectorised envs at different step indices: use the uploaded SSA_F_TRANS_ENV
                                     table (double[E][9], one trans_matrix per environment) instead of M      */
#define SSA_STEP_CATALOG_STATS 0x100 /* ssa_ukf_step / ssa_ukf_step_pinned: append the shard reward reduction of
                                   ssa_ukf_catalog_stats (index offset of its last explicit call) to the step's kernel chain,
                                   inside the same captured graph */
#define SSA_STEP_NO_D2H 0x80    /* ssa_ukf_step_pinned only: do not copy the per-object output block (obs, delta_pos, status)
                                   back to the host; the state stays device-resident and the caller reads what it needs (e.g. the
                                   shard reward terms of ssa_ukf_catalog_stats) */

int ssa_ukf_abi_version(void);
const char* ssa_ukf_last_error(void);
int ssa_ukf_device_count(void);

int ssa_ukf_create(const ssa_ukf_cfg* cfg, int device, ssa_ukf** out);
int ssa_ukf_destroy(ssa_ukf* h);
long ssa_ukf_ld(const ssa_ukf* h); /* leading dimension (padded N) of the device SoA arrays */

/* reset(): host arrays in reference layout. P0 is one 6x6 (p0_per_object = 0) or N of them.     */
int ssa_ukf_reset(ssa_ukf* h, const double* x_true, const double* x_filter, const double* P0,
                  int p0_per_object, void* stream);

/* per-step host inputs: actions int32[E] and/or z_noise double[N][3] (SS2:219-221 draws them at reset) */
int ssa_ukf_upload(ssa_ukf* h, int field, const void* host, size_t bytes, void* stream);
int ssa_ukf_download(ssa_ukf* h, int field, void* host, size_t bytes, void* stream); /* blocks until copied */
/* Every per-step output in ONE device-to-host copy (the drop-in env reads ~16 arrays after each step, SS2:278-322:
 * x_true, x_filter, P_filter, obs, delta_pos/vel, sigma_pos/vel, z_true, y, S, sigmas_h, status, visibility).
 * Layout of `host` (ssa_ukf_snapshot_bytes(h) bytes): double [N][118] = x_true 6 | x_filter 6 | P 36 | obs 12 |
 * delta_pos, delta_vel, sigma_pos, sigma_vel | z_true 3 | y 3 | S 9 | sigmas_h 39; int32 status [N]; uint8 visible
 * [N]; uint8 updated [N].  Blocks until copied.                                                                 */
size_t ssa_ukf_snapshot_bytes(const ssa_ukf* h);
int ssa_ukf_snapshot(ssa_ukf* h, void* host, size_t bytes, void* stream);
/* raw device pointer of a field (device SoA layout) for zero-copy consumers (torch, NCCL) */
int ssa_ukf_device_ptr(ssa_ukf* h, int field, void** dptr, size_t* bytes);

/* The hot path.  M = trans_matrix[i] (row-major GCRS->ITRS).  `flags` selects the fused stages.  */
int ssa_ukf_step(ssa_ukf* h, const double M[9], int flags, void* stream);
/* Same as ssa_ukf_step but brackets each kernel of the step with CUDA events on `stream`, synchronises, and
 * returns the per-kernel durations in milliseconds: ms[0..4] = factor, fx, ut, hx, update (split pipeline) or
 * ms[0] = the fused team kernel.  For measurement only (bench.py roofline of the dominant kernel).            */
int ssa_ukf_step_profile(ssa_ukf* h, const double M[9], int flags, void* stream, double ms[5]);
/* The reference-facing step with HOST buffers (the call an environment makes every step): uploads this step's
 * inputs (actions int32[E] or NULL, z_noise double[N][3] or NULL), runs the step, and copies the step's results
 * back (obs double[N][12], delta_pos double[N], status int32[N]; any may be NULL).  All three phases are
 * asynchronous: inputs/outputs are double-buffered on the device and the copies run on two internal streams, so
 * the H2D of step s+1 and the D2H of step s overlap the kernels of the other step when calls are issued back to
 * back.  Host buffers should be pinned and must stay valid until ssa_ukf_host_join + a synchronize of `stream`
 * (or ssa_ukf_sync).  Results are complete after ssa_ukf_host_join(h, stream) followed by a stream sync.      */
int ssa_ukf_step_host(ssa_ukf* h, const double M[9], int flags, const int32_t* actions_host,
                      const double* z_noise_host, double* obs_host, double* delta_pos_host,
                      int32_t* status_host, void* stream);
/* Pinned-I/O variant of ssa_ukf_step_host for launch-bound batch sizes.  The handle owns two pinned host input
 * blocks and two pinned host output blocks (one per pipeline parity); ssa_ukf_host_io returns their addresses:
 *   inputs   z_noise [N][3], M [9] (the step's trans_matrix[i]), actions [E]
 *   outputs  obs [N][12], delta_pos [N], status [N]
 * The caller fills the inputs of the parity the next call will use (parities alternate 0,1,0,... from the first
 * call; *parity_used reports it), calls ssa_ukf_step_pinned, and reads the outputs of that parity after
 * ssa_ukf_host_join + a synchronize of `stream`.  Per call: ONE host-to-device copy, the step's kernel chain as ONE
 * captured CUDA graph launch (SSA_UKF_GRAPH=0: plain launches), ONE device-to-host copy - the same arithmetic as
 * ssa_ukf_step (the trans_matrix is read from the uploaded block instead of the launch parameters).  Replaces the
 * same reference lines as ssa_ukf_step_host (SS2:259-322, histories SS2:278-322).                               */
int ssa_ukf_host_io(ssa_ukf* h, int parity, double** z_noise, double** M, int32_t** actions, double** obs,
                    double** delta_pos, int32_t** status);
int ssa_ukf_step_pinned(ssa_ukf* h, int flags, void* stream, int* parity_used);
/* With SSA_STEP_CATALOG_STATS a pinned step also reduces the shard's reward terms (reward.py / SS2:324-354 over the
 * whole shard: the 5 doubles of SSA_F_CATALOG_STATS) into the device slot of ITS parity and copies them to the pinned
 * host block of that parity on the internal download stream - the caller's stream never waits for a read-back, and a
 * consumer (host, or an NCCL gather on a side stream) may still read step s while step s + 1 runs.  Returns the two
 * addresses of `parity`: host (valid after ssa_ukf_host_join + synchronize) and device.                         */
int ssa_ukf_host_stats(ssa_ukf* h, int parity, double** stats_host, double** stats_device);
/* ---- device-resident episodic mode (vectorised reset, SURVEY 8f-2) ---------------------------------------------
 * Replaces, for E parallel environments, the whole host side of an RL step: reset() with its catalog sampling and
 * noise draws (SS2:193-241), the per-step bookkeeping of step() (SS2:243-367: step counter, trans_matrix[i],
 * z_noise[i], update_interval gate SS2:292, reward / done SS2:324-354) and the auto-reset of finished episodes.
 * Random numbers are counter-based (Philox4x32-10 keyed by the environment's seed, addressed by episode / object /
 * step - csrc/ssa_rng.h): same distributions as the reference, NOT the same streams as its np_random (the host-RNG
 * path ssa_ukf_reset + ssa_ukf_step keeps stream parity).  'shaped' rewards are not available here.
 *   rollout_config  catalog [n_orbits][6], trans_matrix table [n_table][9] (row i = step i), one 64-bit seed per env,
 *                   x_sigma[6], z_sigma[3] (radians / metres), P0[36], update_interval
 *   rollout_io      pinned host blocks owned by the handle: actions [E] (in); obs [N][12], reward [E],
 *                   greedy [E][SSA_N_TASKERS], done [E] (out)
 *   rollout_reset   draw every environment, step index 0; outputs: obs, greedy
 *   rollout_step    one step of every environment with the actions in the pinned block: ONE H2D copy, ONE CUDA-graph
 *                   launch (noise, the five UKF kernels, reward / done, reset of the finished environments and their
 *                   fresh obs when auto_reset, greedy taskers of the new state), ONE D2H copy.  Asynchronous on
 *                   `stream`; outputs are valid after a synchronize.  With auto_reset the obs rows of a finished
 *                   environment are those of its NEW episode; reward / done refer to the step just taken.        */
int ssa_ukf_rollout_config(ssa_ukf* h, const double* orbits, int n_orbits, const double* trans_table, int n_table,
                           const uint64_t* seeds, const double x_sigma[6], const double z_sigma[3], const double P0[36],
                           int update_interval);
int ssa_ukf_rollout_io(ssa_ukf* h, int32_t** actions, double** obs, double** reward, int32_t** greedy, uint8_t** done);
int ssa_ukf_rollout_reset(ssa_ukf* h, void* stream);
/* auto_reset bit 0: re-draw finished environments inside the step; bit 1 (SSA_ROLLOUT_DEVICE_IO): no host copies —
 * the actions are read from the device buffer SSA_F_ROLLOUT_ACTIONS and obs / reward / done / greedy stay in the device
 * block (SSA_F_ROLLOUT_*), for a policy that lives on the same GPU (everything stream-ordered, nothing synchronises). */
#define SSA_ROLLOUT_DEVICE_IO 2
/* bit 2 (SSA_ROLLOUT_OBS_F32): the observations leave the device as float32 (rounded to nearest, numpy's
 * astype(float32)): the last kernel of the step's graph writes obs [N][12] as floats and the D2H copy moves those
 * 48 N bytes (+ the reward / greedy / done tail) instead of 96 N — for a learner that casts its observations to float32
 * anyway (RLlib's preprocessors do, rl_agents/RLLib_PPO_training.py).  The float64 rows stay valid on the device.    */
#define SSA_ROLLOUT_OBS_F32 4
int ssa_ukf_rollout_step(ssa_ukf* h, int auto_reset, void* stream);
/* the float32 observation blocks of SSA_ROLLOUT_OBS_F32: pinned host mirror and device block, [N][12] floats          */
int ssa_ukf_rollout_obs_f32(ssa_ukf* h, float** host, float** device);
/* make `stream` wait for every outstanding internal copy of ssa_ukf_step_host / ssa_ukf_step_pinned */
int ssa_ukf_host_join(ssa_ukf* h, void* stream);
/* Convenience wrappers with the reference's call structure */
int ssa_ukf_predict(ssa_ukf* h, void* stream);                      /* truth + predict              */
int ssa_ukf_update(ssa_ukf* h, const double M[9], int all, void* stream); /* update (all | actions[e]) + epilogue */

/* per-environment reductions: reward / done (SS2:324-354) and the greedy taskers (agents.py).
 * step_index = i after the increment of SS2:259; a negative step_index selects the uploaded per-env
 * SSA_F_STEP_INDEX table.  The step index also keys SSA_TASKER_SHANNON's determinant history (see there).  'shaped' rewards need the reward history: the device returns ENV_STATS and the
 * host finishes them (SS2:339-351).                                                                       */
int ssa_ukf_env_reduce(ssa_ukf* h, const double M[9], int step_index, void* stream);
/* reward.py score terms from the current covariances: out double[N][6] =
 * [score_scaled_trace_P, score_trace_P, score_scaled_det_P(dt), score_det_P, score_det_pos_P, |dpos|] */
int ssa_ukf_scores(ssa_ukf* h, void* stream);
/* Catalog generator (SURVEY 8f-4): the acceptance rule of envs/orbit_gen.py:47-75 for a batch of K candidate orbits
 * (GCRS states at the epoch).  For each candidate and each of the n sample times i*step_s: two-body propagation from
 * the epoch (the reference uses fx_xyz_markley there; this is the same two-body flow through ssa_fx), geodetic
 * altitude of x @ trans_table[i] (ecef2lla, transformations.py:239-279) and elevation of hx_aer_erfa; accepted iff
 * every altitude > min_alt and either the object is always visible, or it is seen within the first
 * `first_window` samples and no visibility gap reaches `max_gap` samples.  Stand-alone (no handle): host arrays in,
 * accept[K] out (and, optionally, elev / alt [K][n] for inspection).                                              */
int ssa_orbit_gen_eval(const double* cand, int K, const double* trans_table, int n, double step_s, const double obs_itrs[3],
                       const double T[9], double obs_limit, double min_alt, int first_window, int max_gap, uint8_t* accept,
                       double* elev, double* alt, int device);
/* HOST (no device): the GCRS -> ITRS rotation table the path takes as its per-step input — trans_matrix[i] of
 * ssa_tasker_simple_2.py:136-137, which the reference builds through ERFA (envs/transformations.py:143-214) — for the n
 * UTC instants (year-month-day, seconds_of_day) + i * dt (whole seconds are used, like the reference's datetime fields).
 * ERFA-free restatement (csrc/ssa_frames.h): exact calendar, leap seconds, Earth rotation angle, TIO locator and polar
 * motion; CIP X, Y from the IAU 2006/2000A series truncated at 1 mas (7.5e-9 rad against the SOFA matrix of the
 * reference's tests.py:107-109).  eop: daily IERS rows [mjd, x", y", UT1-UTC s, dX", dY"] (n_eop of them) or NULL.
 * out: [n][9] row-major matrices.                                                                                     */
int ssa_trans_matrix_table(int year, int month, int day, double seconds_of_day, double dt, int n, const double* eop, int n_eop,
                           double* out);
/* Catalog mode (C4: one shard of a large catalog per GPU): the shard's reward terms over ALL its objects, left in
 * device memory (SSA_F_CATALOG_STATS, 5 doubles) so that the shards can be combined with one small all_gather:
 * max delta_pos (SS2:329-331), sum of the trinary counts (results.py:431-433) and the object count, the largest
 * trace P and its index + index_offset (agents.py:8, first maximum wins).                                        */
int ssa_ukf_catalog_stats(ssa_ukf* h, long index_offset, void* stream);
/* Consistency diagnostics of the current state (SURVEY 8f-3): per object NEES = (x_true - x)^T P^-1 (x_true - x)
 * (SS2:436-446 anees), and for the objects updated by the last step run with SSA_STEP_RECORD the NIS
 * y^T S^-1 y (SS2:564-569) and the innovation-bound flags (SS2:598-604) -> SSA_F_DIAG, SSA_F_INNOV_FLAGS.      */
int ssa_ukf_diagnostics(ssa_ukf* h, void* stream);
/* Innovation whiteness statistics of B innovation series (SURVEY 8f-3): y [n_series][n][3] with a validity mask
 * valid [n_series][n] (an observation was taken at that step / the object was the tasked one), host buffers in and out.
 *   dw  [n_series][3]            Durbin-Watson statistic over the valid entries in order     SS2:782-832 innovation_dw_test
 *   acf [n_series][3][nlags+1]   autocorrelation, statsmodels acf(missing='conservative')    SS2:655-668 autocorrelation    */
int ssa_innovation_stats(const double* y, const uint8_t* valid, int n_series, int n, int nlags, double* dw, double* acf, int device);

int ssa_ukf_sync(ssa_ukf* h, void* stream);
/* number of kernel launches issued through this handle so far (bench.py `gpu_launches`) */
long ssa_ukf_launch_count(const ssa_ukf* h);

/* FP64 pipe microbenchmark (dependent DFMA chains on every SM) used as the roofline denominator:
 * returns achieved TFLOP/s (2 flop per DFMA), timed with CUDA events on `stream`.                  */
int ssa_ukf_fp64_peak(int device, void* stream, double* tflops);

/* ---- operator-level entry points -----------------------------------------------------------------
 * The reference's plug points are Python callables handed to filterpy through env_config
 * (envs/__init__.py:27-28: fx, hx, mean_z, residual_z, msqrt).  These evaluate the DEVICE build of
 * the same operators on host arrays (synchronous; n independent evaluations, one GPU thread each), so
 * that calling an operator directly runs the code the fused kernel runs.  Also used by the parity
 * tests to compare sm_100a with the host twin function by function.                                  */
/* op: 0 sin 1 cos 2 tan 3 atan 4 asin 5 acos 6 exp 7 log 8 sinh 9 cosh 10 tanh 11 atanh 12 asinh
 *     13 acosh 14 x^(2/3) 15 atan2(a,b) 16 python a%b 17 a/b 18 sqrt                                  */
int ssa_unit_math(int op, const double* a, const double* b, double* out, int n, int device);
/* fx_xyz_farnocchia (envs/farnocchia.py:1053): x[n][6] -> out[n][6]; exc[n] != 0 where numba would raise */
int ssa_unit_fx(const double* x, double dt, double* out, int32_t* exc, int n, int device);
/* hx_aer_erfa (envs/dynamics.py:219): x[n][stride] (first 3 used) -> out[n][3] = az, el, range      */
int ssa_unit_hx_aer(const double* x, int stride, const double M[9], const double obs_itrs[3], const double T[9],
                    double* out, int n, int device);
/* op 0: aer2uvw  1: uvw2aer  2: residual_z_aer(a, b)   (transformations.py:283-316, dynamics.py:260) */
int ssa_unit_aer(int op, const double* a, const double* b, double* out, int n, int device);
/* robust_cholesky(lam * P) (envs/dynamics.py:402): packed upper [n][21] in/out; ret = attempt or -1  */
int ssa_unit_robust_chol(const double* P_packed, double lam, double* U_packed, int32_t* ret, int n, int device);
/* numpy.linalg.inv of 3x3 (filterpy UKF.update SI = inv(S))                                          */
int ssa_unit_inv3(const double* S, double* SI, int32_t* ok, int n, int device);

#ifdef __cplusplus
}
#endif
#endif /* SSA_UKF_H */
