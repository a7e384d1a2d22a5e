/* rdv_b200.h -- C ABI of librdv_b200.so: the B200 (sm_100a) batched replacement for the
 * RendezvousEnv step()/reset() hot path of cfdeinza/reinforcement-learning-rendezvous.
 *
 * Boundary rules
 *   - extern "C", plain pointers and sizes only; no C++/torch types cross this line.
 *   - Every buffer is owned by the caller (PyTorch CUDA tensors in the Python host);
 *     the library never allocates, frees or keeps device memory after a call returns.
 *   - All entry points enqueue work on the caller's stream and return immediately
 *     (no device synchronisation inside); 0 = success, negative = RdvStatus error.
 *   - Results are a pure function of (params, state, actions, seed, env_offset,
 *     episode index): independent of grid shape and of how envs are sharded over GPUs.
 *   - There is no CPU fallback: on a machine without a usable GPU the calls return
 *     RDV_ERR_CUDA.
 *
 * Each entry point cites the reference interface (file:line under /root/reference)
 * it replaces.
 */
#ifndef RDV_B200_H
#define RDV_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RDV_ABI_VERSION 16
#define RDV_OBS_DIM 17          /* rendezvous_env.py:133-137 Box(-1, 1, (17,), float32) */
#define RDV_ACT_DIM 6           /* rendezvous_env.py:140-144 Box(-1, 1, (6,),  float32) */
#define RDV_N_UNIFORMS 24       /* draws consumed by one reset(): rendezvous_env.py:229-250 */

/* Rows of RdvState.f64 ([RDV_NF64][ld], structure-of-arrays, one column per env). */
enum {
    RDV_RCX = 0, RDV_RCY, RDV_RCZ,            /* rc: chaser position, LVLH [m]            */
    RDV_VCX, RDV_VCY, RDV_VCZ,                /* vc: chaser velocity, LVLH [m/s]          */
    RDV_QCW, RDV_QCX, RDV_QCY, RDV_QCZ,       /* qc: chaser attitude (scalar first)       */
    RDV_WCX, RDV_WCY, RDV_WCZ,                /* wc: chaser rate, chaser body frame       */
    RDV_QTW, RDV_QTX, RDV_QTY, RDV_QTZ,       /* qt: target attitude                      */
    RDV_WTX, RDV_WTY, RDV_WTZ,                /* wt: target rate, target body frame       */
    RDV_TDV, RDV_TDW,                         /* total_delta_v / total_delta_w (:201-202) */
    RDV_EPRET,                                /* return of the running episode (Monitor 'r') */
    RDV_NF64
};
/* Rows of RdvState.i32 ([RDV_NI32][ld]). t = round(step*dt, 3) and the bubble radius
 * max(bubble0 - step*rate, bubble_min) are derived from RDV_I_STEP (:193-198). */
enum { RDV_I_STEP = 0, RDV_I_SUCCESS, RDV_I_COLLIDED, RDV_I_EPISODE, RDV_NI32 };

/* Slots of the device statistics vector (double[RDV_NSTATS], accumulated with atomics). */
enum {
    RDV_S_STEPS = 0, RDV_S_EPISODES, RDV_S_RETURN, RDV_S_LENGTH, RDV_S_SUCCEEDED, RDV_S_COLLIDED,
    RDV_S_DELTA_V, RDV_S_DELTA_W,
    RDV_S_END_OBS, RDV_S_END_TIME, RDV_S_END_BUBBLE, RDV_S_END_ATTITUDE,   /* :377 end reasons */
    RDV_S_REWARD, RDV_S_RK_ACCEPTED, RDV_S_RK_REJECTED, RDV_S_FAILURES,
    RDV_NSTATS
};

/* Columns of the per-episode record written for envs whose episode just ended. */
enum { RDV_EP_RETURN = 0, RDV_EP_LENGTH, RDV_EP_SUCCESS, RDV_EP_COLLIDED, RDV_EP_DELTA_V, RDV_EP_DELTA_W,
       RDV_EP_NCOL };

typedef enum RdvStatus {
    RDV_OK = 0,
    RDV_ERR_NULL = -1,        /* a required pointer is NULL                          */
    RDV_ERR_SIZE = -2,        /* n < 0, ld < n, or a bad enum value                  */
    RDV_ERR_ALIGN = -3,       /* a pointer is not aligned for its vector access      */
    RDV_ERR_PARAMS = -4,      /* rdv_params_derive rejected the configuration        */
    RDV_ERR_CUDA = -5,        /* kernel launch / CUDA runtime failure                */
    RDV_ERR_UNSUPPORTED = -6
} RdvStatus;

/* Integrator used for the two attitude propagations (rendezvous_env.py:552-604). */
enum {
    RDV_INTEGRATOR_RK45 = 0,       /* adaptive Dormand-Prince replica of scipy solve_ivp(RK45) */
    RDV_INTEGRATOR_CLOSED_FORM = 1 /* exact torque-free isotropic rotation; opt-in, gated      */
};

/* Environment constants.  The first block mirrors the RendezvousEnv constructor
 * (rendezvous_env.py:17-70) and reward_kwargs (:313); fill it (or start from
 * rdv_params_default) and call rdv_params_derive, which fills the second block
 * exactly as the constructor does (:75-126).  Passed BY VALUE to the kernels. */
typedef struct RdvParams {
    /* ---- inputs ---- */
    double rc0[3], vc0[3], qc0[4], wc0[3], qt0[4], wt0[3];      /* nominal initial state        */
    double rc0_range, vc0_range, qc0_range, wc0_range, qt0_range, wt0_range;
    double koz_radius, corridor_half_angle, h, dt, t_max;
    double collision_coef, bonus_coef, fuel_coef, att_coef;     /* get_bubble_reward kwargs     */
    double inertia_c[9], inertia_t[9];                          /* row-major 3x3 (:75-79,:96-100) */
    double torque_c[3];                                         /* held chaser torque (env: 0)  */
    int32_t integrator;                                         /* RDV_INTEGRATOR_*             */
    int32_t reserved0;
    /* ---- derived by rdv_params_derive ---- */
    double inv_inertia_c[9], inv_inertia_t[9];
    double max_delta_v, max_delta_w, max_axial_distance, max_axial_speed, max_wc;
    double max_attitude_error, max_rd_error, max_vd_error, max_qd_error, max_wd_error;
    double rd[3], capture_axis[3], corridor_axis[3];
    double bubble0, bubble_rate, bubble_min, n;
    double cw[17];                 /* non-zero entries of the CW transition matrix (dynamics.py:40-47) */
    float max_delta_v_f32;         /* fp32 constants used when actions are float32 (NumPy-2 promotion) */
    float fuel_num_f32;            /* (float)(dt*fuel_coef)                                            */
    float fuel_den_f32;            /* (float)(3*max_delta_v)                                           */
    int32_t iso_c, iso_t;          /* 1: inertia = c*Identity and zero torque -> rate is constant      */
    int32_t done_steps;            /* smallest step count k with round(k*dt, 3) >= t_max (:193, :369)   */
    /* reciprocals / squares / products of the constants above, so the per-step path has no division */
    double inv_max_attitude_error, inv_max_rd_error, inv_max_qd_error;
    double koz_radius_sq, max_rd_error_sq, max_vd_error_sq, max_wd_error_sq;
    double fuel_scale;             /* dt*fuel_coef / (3*max_delta_v)   (:333)                          */
    double att_scale, bonus_scale, collision_scale;   /* dt*att_coef, dt*bonus_coef, dt*collision_coef  */
    double obs_inv_r, obs_inv_v, obs_inv_w;           /* 1/(2*max_axial_distance), 1/(2*5), 1/(2*max_wc) */
    double near_sq;                /* max(koz, |rd| + max_rd_error)^2 (+margin): beyond it neither a collision,
                                    * a success nor a reward bonus is possible (:397, :417, :348)        */
    int32_t box_hi_r, box_hi_v, box_hi_w;   /* high words of max_axial_distance / max_axial_speed / max_wc times  *
                                             * (1 - 1e-6): the fast path of the observation Box test (:367)       */
    int32_t reserved1;
} RdvParams;

/* Environment state: device pointers into caller-owned buffers. */
typedef struct RdvState {
    double  *f64;     /* [RDV_NF64][ld] */
    int32_t *i32;     /* [RDV_NI32][ld] */
    int64_t  ld;      /* leading dimension (>= n), in elements */
    /* Per-env parameter batches (the sensitivity-sweep axes of sensitivity_analysis.py:97-134 as ONE batch): a
     * device array of derived RdvParams and, for every block of 32 consecutive envs, the index of the entry its envs
     * use.  NULL: every env uses the RdvParams passed to the call.  With a table the call's RdvParams only selects the
     * kernel family (all entries must share iso_c / iso_t / integrator with it); supported for the reference's
     * isotropic bodies with the RK45 integrator. */
    const struct RdvParams *param_table;   /* nullable, device, [entries]                       */
    const int32_t *param_block;            /* device, [ceil(n / 32)]: entry of envs 32 b .. 32 b + 31 */
} RdvState;

/* Inputs/outputs of one batched step.  Nullable members are marked. */
typedef struct RdvStepIO {
    const void *actions;     /* [n][6] row-major, float32 (act_f64 = 0) or float64 (act_f64 = 1)  */
    int32_t  act_f64;
    int32_t  auto_reset;     /* 0: off.  1: envs that finish are reset by the same call (VecEnv semantics)  */
    float   *obs;            /* [n][17] observation after the step (after the reset if auto-reset) */
    double  *reward;         /* [n]                                                                */
    uint8_t *done;           /* [n]                                                                */
    float   *terminal_obs;   /* nullable [n][17]: last observation of finished episodes only       */
    int8_t  *end_reason;     /* nullable [n]: -1 running, 0 obs, 1 time, 2 bubble, 3 attitude      */
    double  *episode_record; /* nullable [n][RDV_EP_NCOL]: written for finished episodes only      */
    double  *stats;          /* nullable [RDV_NSTATS] device accumulator                           */
    /* -- one-copy host path (RendezvousVecEnv): everything a VecEnv step returns, in one caller-owned block -- */
    float   *reward_f32;     /* nullable [n]: the reward rounded to float32 (what SB3's VecEnv returns)        */
    int32_t *fin_count;      /* nullable [1]: number of rows appended to fin_rows by this call; the library     *
                              * zeroes it on the stream before the launch                                       */
    void    *fin_rows;       /* nullable [fin_capacity] RdvFinishedRow: one row per env whose episode ended in  *
                              * this call, in no particular order (sort by .env on the host if needed)          */
    int32_t  fin_capacity;   /* rows fin_rows can hold (n is always enough)                                     */
    int32_t  fin_append;     /* 1: keep fin_count and append (a further launch of the same step, other env range) */
    int32_t  fin_env_base;   /* added to the env index stored in the rows (index of env 0 of this launch)       */
    int32_t  reserved;
} RdvStepIO;

/* What a VecEnv's info dict of a finished env carries (DummyVecEnv.step_wait + Monitor.step, main.py:33-34):
 * the env index, the end reason of get_done_condition (rendezvous_env.py:377), the terminal observation and the
 * episode record.  128 bytes, 16-byte aligned. */
typedef struct RdvFinishedRow {
    int32_t env;                         /* local env index                                   */
    int32_t end_reason;                  /* 0 obs, 1 time, 2 bubble, 3 attitude               */
    float   terminal_obs[RDV_OBS_DIM];   /* last observation of the episode (pre-reset)       */
    float   pad;
    double  record[RDV_EP_NCOL];         /* RDV_EP_* columns                                  */
} RdvFinishedRow;

/* -- constants ------------------------------------------------------------------------------ */
int  rdv_abi_version(void);
int  rdv_sizeof_params(void);
/* sizeof of the ABI structs as this build sees them (a binding checks its own mirrors against these):
 * 0 RdvParams, 1 RdvState, 2 RdvStepIO, 3 RdvRolloutIO, 4 RdvPolicy, 5 RdvFinishedRow; -1 for anything else. */
int  rdv_sizeof(int which);
const char *rdv_strerror(int status);

/* Defaults of RendezvousEnv.__init__ (rendezvous_env.py:17-70). */
void rdv_params_default(RdvParams *p);
/* Derived constants of RendezvousEnv.__init__ (rendezvous_env.py:75-126) and the CW matrix of
 * clohessy_wiltshire_solution (utils/dynamics.py:40-47).  Returns RDV_ERR_PARAMS when the
 * constructor's assertions (:155-156) would fail or a matrix is singular. */
int  rdv_params_derive(RdvParams *p);

/* -- the hot path ------------------------------------------------------------------------------ */
/* RendezvousEnv.step (rendezvous_env.py:160-221) for n envs, plus the auto-reset that SB3's
 * DummyVecEnv.step_wait performs around it (main.py:33-34).  env_offset is the global index
 * of env 0 of this shard (Philox key for resets). */
int rdv_step(const RdvParams *p, const RdvState *s, const RdvStepIO *io, int64_t n,
             uint64_t seed, int64_t env_offset, void *cuda_stream);

/* fp32 tanh MLP obs[17] -> hidden -> hidden -> action[6] of an SB3 MlpPolicy (main.py:39-48), deterministic mean
 * clipped to [-1,1] (model.predict, monte_carlo.py:128-133).  Weights are row-major [out][in] as in torch.nn.Linear. */
typedef struct RdvPolicy {
    const float *w0, *b0;    /* [H][17], [H] */
    const float *w1, *b1;    /* [H][H],  [H] */
    const float *w2, *b2;    /* [6][H],  [6] */
    int32_t hidden;          /* H, must be 64 */
    int32_t reserved;
    const float *log_std;    /* nullable [6]: state-independent log std of the Gaussian head (sampling mode) */
} RdvPolicy;
/* K consecutive steps of every env in one launch (state stays in registers; finished envs are reset in
 * place).  This is the rollout-collection loop of SB3's collect_rollouts around env.step
 * (main.py:114 -> OnPolicyAlgorithm.collect_rollouts) with the action taken from `actions` or drawn on the
 * device.  The per-step results a rollout buffer needs are optional outputs. */
enum { RDV_ACTIONS_F32 = 0, RDV_ACTIONS_F64 = 1, RDV_ACTIONS_PHILOX = 2,
       RDV_ACTIONS_POLICY = 3,          /* a = clip(actor(obs)): model.predict(deterministic=True)                 */
       RDV_ACTIONS_POLICY_SAMPLE = 4 }; /* a ~ N(actor(obs), exp(log_std)^2), the env gets clip(a) and actions_out  *
                                         * the unclipped draw: SB3 collect_rollouts (noise: Philox(action_seed; env  *
                                         * id, step_base + k), Box-Muller in float32)                               */
typedef struct RdvRolloutIO {
    int32_t  steps;          /* K                                                                          */
    int32_t  action_source;  /* RDV_ACTIONS_*                                                              */
    int32_t  auto_reset;     /* 1: VecEnv semantics (finished envs restart inside the launch)              */
    int32_t  reserved;       /* set to 0 (the library passes its reset-prefetch period to the kernel here)   */
    const void *actions;     /* [K][n][6] float32 / float64 for the tensor sources                         */
    uint64_t action_seed;    /* RDV_ACTIONS_PHILOX: U(-1,1) fp64 actions from Philox(action_seed; global   */
    int64_t  step_base;      /*   env id, step_base + k): six 32-bit draws per env-step, a = (w + 0.5) 2^-31 - 1 */
    double  *actions_out;    /* nullable [K][n][6]: the applied Philox (float64) or policy (float32!) actions */
    float   *obs;            /* [n][17] observation after the last step (post-reset for finished envs)     */
    double  *rewards;        /* nullable [K][n]                                                            */
    uint8_t *dones;          /* nullable [K][n]                                                            */
    float   *obs_steps;      /* nullable [K][n][17] observation returned by every step                     */
    double  *stats;          /* nullable [RDV_NSTATS] device accumulator                                   */
    RdvPolicy policy;        /* RDV_ACTIONS_POLICY: a = clip(actor(obs)), evaluated in the launch (tensor cores) */
    /* Caller-owned scratch that carries every env's prefetched NEXT reset state (rendezvous_env.py:223-270 for
     * (env, episode + 1): it depends on the seed and the counters only, not on the trajectory) from one launch to
     * the next, so that short launches run at the rate of long ones.  [RDV_RESET_ROWS][ld] like RdvState.f64, offset
     * to the same env; rows 0..19 state, 20 / 21 the collided / success flags, row 22 the episode index the row was
     * computed for (0 = none; a row is used only if it equals the env's episode + 1).  Zero row 22 whenever the
     * seed or the parameters change.  NULL: the rows live and die with the launch. */
    double  *reset_rows;
    int32_t  sm_reserve;     /* SMs left without a CTA of this launch, e.g. 1 so that the statistics all-reduce of the *
                              * previous rollout (another stream) runs beside it instead of behind it                  */
    int32_t  reserved2;
    /* Monte-Carlo evaluator mode (monte_carlo.py:94-207), needs auto_reset = 0: [n][RDV_MC_NCOL] per-episode
     * results accumulated in registers from the state at launch (sample 0) to the env's first done; finished envs
     * stop stepping.  NULL: off. */
    double  *mc_out;
    /* Policy tables (many actors in one launch, e.g. one model per parameter set of a sweep): a device array of
     * RdvPolicy entries and, for every tile of 128 consecutive envs, the index of the entry its envs use.  NULL: every
     * env uses `policy`, exactly as without the fields.  With a table `policy` is not read (its weights may be NULL);
     * needs a policy action source (RDV_ACTIONS_POLICY / _SAMPLE, every entry with log_std for sampling) and the
     * reference's isotropic bodies with the RK45 integrator; combines with the evaluator mode, auto-reset, reset_rows
     * and RdvState.param_table.  Every entry must have hidden = 64 and non-NULL weights and biases, and, for
     * RDV_ACTIONS_POLICY_SAMPLE, a non-NULL log_std; the library does not read the table on the host, so the kernel
     * checks each entry when a group stages it.  A tile whose index lies outside [0, policy_count), or whose entry
     * fails that check, takes zero actions, and each of its env-steps counts in RDV_S_FAILURES. */
    const RdvPolicy *policy_table;    /* nullable, device, [policy_count]                                  */
    const int32_t *policy_tile;       /* device, [ceil(n / 128)]: entry of envs 128 t .. 128 t + 127        */
    int32_t  policy_count;
    int32_t  reserved3;
} RdvRolloutIO;
#define RDV_RESET_ROWS 23
/* Columns of RdvRolloutIO.mc_out: the workbook columns of monte_carlo.py:190-203 (errors in rad / rad/s, the host
 * converts to degrees; ep_len in steps), then what else an evaluator wants. */
enum { RDV_MC_EP_LEN = 0, RDV_MC_NUM_COLLISIONS, RDV_MC_COLLIDED, RDV_MC_TOTAL_REWARD, RDV_MC_TOTAL_DELTA_V,
       RDV_MC_NUM_SUCCESSES, RDV_MC_SUCCEEDED, RDV_MC_MIN_KOZ, RDV_MC_POS_ERR, RDV_MC_VEL_ERR, RDV_MC_ATT_ERR,
       RDV_MC_ROT_ERR, RDV_MC_LEVEL,      /* constraints met at the averaging start: 0 all four .. 3 position only, 4 none */
       RDV_MC_TAIL_COUNT,                 /* samples averaged                                                   */
       RDV_MC_END_REASON,                 /* -1: still running when the launch ended                             */
       RDV_MC_TOTAL_DELTA_W, RDV_MC_NCOL };
int rdv_rollout(const RdvParams *p, const RdvState *s, const RdvRolloutIO *io, int64_t n, uint64_t seed,
                int64_t env_offset, void *cuda_stream);

/* Columns of the trajectory record of rdv_rollout_trajectory.  Columns 0 .. RDV_NF64 - 1 are the rows of RdvState.f64
 * in their order (state, totals, episode return); then the RdvState.i32 rows as doubles; then what rdv_errors returns
 * for that state: get_errors (position [m], velocity [m/s], attitude [rad], rate [rad/s]), dist_from_koz, and
 * check_collision / check_success (with the sticky collided flag) as 0 / 1. */
enum { RDV_TR_I_STEP = RDV_NF64, RDV_TR_I_SUCCESS, RDV_TR_I_COLLIDED, RDV_TR_I_EPISODE,
       RDV_TR_POS_ERR, RDV_TR_VEL_ERR, RDV_TR_ATT_ERR, RDV_TR_ROT_ERR, RDV_TR_KOZ, RDV_TR_COLLISION, RDV_TR_SUCCESS,
       RDV_TR_NCOL };
/* rdv_rollout that also records the fp64 trajectory: traj [K][RDV_TR_NCOL][n] (8-byte aligned, 272 bytes per
 * env-step), element (k, col, i) at traj[(k * RDV_TR_NCOL + col) * n + i].  Row k is env i after step k's propagation
 * and evaluation and BEFORE an auto-reset (for an env that finished at step k: its terminal state); columns
 * 0 .. RDV_TR_I_EPISODE hold what RdvState would hold there, the rest what rdv_errors returns on that state, bit for
 * bit.  In the evaluator mode a finished env stops stepping, and its later rows repeat its last one.  Every other
 * output is the same as rdv_rollout's for the same arguments (which it accepts and checks in the same way);
 * traj NULL: RDV_ERR_NULL. */
int rdv_rollout_trajectory(const RdvParams *p, const RdvState *s, const RdvRolloutIO *io, double *traj, int64_t n,
                           uint64_t seed, int64_t env_offset, void *cuda_stream);

/* RendezvousEnv.reset (rendezvous_env.py:223-270) for the envs selected by mask (NULL = all).
 * The 24 uniform draws come from Philox4x32-10 keyed by (seed; env_offset+i, episode index),
 * or from `uniforms` ([n][24], in [0,1)) when it is not NULL (test hook that pins the
 * draw order against the reference).  bump_episode: 1 increments the episode index first. */
int rdv_reset(const RdvParams *p, const RdvState *s, const uint8_t *mask, const double *uniforms,
              float *obs, int64_t n, uint64_t seed, int64_t env_offset, int bump_episode,
              void *cuda_stream);

/* RendezvousEnv.get_observation (rendezvous_env.py:294-311). */
int rdv_observe(const RdvParams *p, const RdvState *s, float *obs, int64_t n, void *cuda_stream);

/* get_errors / check_collision / check_success / dist_from_koz (rendezvous_env.py:388-468,
 * :510-537) -- what monte_carlo.evaluate and the callbacks read after every step.
 * errors [n][4]; collision, success [n] (success honours the sticky collided flag); koz [n]. */
int rdv_errors(const RdvParams *p, const RdvState *s, double *errors, uint8_t *collision,
               uint8_t *success, double *koz, int64_t n, void *cuda_stream);

/* After a caller overwrote the state (monte_carlo.py:106-112 does), optionally recompute the
 * sticky collided / success flags the way reset() does (:260-261).  The reference evaluator
 * does NOT do this; it is provided for callers that want consistent flags. */
int rdv_refresh_flags(const RdvParams *p, const RdvState *s, int64_t n, void *cuda_stream);

/* chaser2lvlh / target2lvlh (transpose = 0: out = R(q) v) and lvlh2chaser / lvlh2target
 * (transpose = 1: out = R(q)^T v) of rendezvous_env.py:470-508, with quat2mat's
 * re-normalisation (utils/quaternions.py:48-68).  q [n][4], v [n][3], out [n][3], device fp64. */
int rdv_frame_transform(const double *q, const double *v, double *out, int64_t n, int transpose,
                        void *cuda_stream);

/* -- stand-alone policy forward (model.predict of an SB3 MlpPolicy, monte_carlo.py:128-133) ----------------
 * obs [n][17] float32 -> actions [n][6] float32, deterministic mean clipped to [-1,1].
 * rdv_policy_forward: tcgen05 tensor-core kernel (TMEM accumulators, every product as three MMAs of fp16 halves = fp32-level accuracy).
 * rdv_policy_forward_ffma: the same op as plain fp32 FMAs, one thread per env (numerics reference). */
int rdv_policy_forward(const RdvPolicy *pi, const float *obs, float *actions, int64_t n, void *cuda_stream);
int rdv_policy_forward_ffma(const RdvPolicy *pi, const float *obs, float *actions, int64_t n, void *cuda_stream);

/* Development / test knobs that used to be environment variables (read once at load as defaults); every setting gives
 * the same bits.  Returns the previous value, or RDV_ERR_SIZE for an unknown key.
 *   RDV_TUNE_ROLLOUT_TPB      forces the rollout CTA size (256 | 384 | 448 | 512, 0 = automatic)
 *   RDV_TUNE_RESET_REFILL     reset prefetch period in steps (0 = reset on demand only; default 12)
 *   RDV_TUNE_ROLLOUT_PDL      1 (default): rdv_rollout launches with programmatic stream serialisation, so the
 *                             prologue of a launch overlaps the tail of the previous kernel; 0: plain launch
 *   RDV_TUNE_ROLLOUT_HELPERS  1 (default): launches of 385..448 envs per SM in one pass (65,536 envs on a B200) run
 *                             with two helper warps per CTA that recompute the used reset rows beside the 14 worker
 *                             warps; 0: the workers refill their rows themselves every RESET_REFILL steps */
enum { RDV_TUNE_ROLLOUT_TPB = 0, RDV_TUNE_RESET_REFILL = 1, RDV_TUNE_ROLLOUT_PDL = 2, RDV_TUNE_ROLLOUT_HELPERS = 3 };
int rdv_tune(int key, int value);

/* Test hook: y[i] = f(x[i]) for the device math helpers the step is built from.  op 0: 1/sqrt(x), 1: 1/x,
 * 2: sqrt(x), 3: x^-0.1 (fp64 controller), 4: x^-0.1 (float32 controller), 5: acos(round(x, 5))
 * (angle_between_vectors, utils/general.py:163-181); at x = s^2 > 0, one attempted step of the plane attitude solver:
 * 6-9: P, Q, R, I of rdv_plane_poly.h, 10-13: the same four from the stagewise attempt. */
int rdv_math_probe(const double *x, double *y, int64_t n, int op, void *cuda_stream);

/* Measured-peak helper for the roofline: runs `iters` dependent-chain-free DFMA per thread on
 * every SM and writes one double per thread to `sink` ([blocks*threads]).  flops = 2*iters*16*
 * blocks*threads. */
int rdv_fp64_peak_probe(double *sink, int blocks, int threads, int iters, void *cuda_stream);

#ifdef __cplusplus
}
#endif
#endif /* RDV_B200_H */
