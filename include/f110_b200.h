/*
 * f110_b200.h -- C ABI of the B200-native batched F1TENTH step path (libf110_b200.so).
 *
 * The reference (ahoop004/f110_gymnasium_ros2_jazzy) has no FFI: its step path is Python +
 * numba behind two Python classes.  This header is the boundary a native backend for those
 * classes binds to; each entry point names the reference interface it replaces.  Paths are
 * relative to f110_gymnasium/gym/f110_gym/envs/ in the reference tree.
 *
 *   Simulator.__init__            base_classes.py:478-510   -> f110_create
 *   Simulator.set_map             base_classes.py:512-524   -> f110_set_map (+ f110_set_tables)
 *     ScanSimulator2D.__init__    laser_models.py:360-381      (sin/cos tables, increments)
 *     ScanSimulator2D.set_map     laser_models.py:383-427      (dt = resolution * EDT, host side)
 *   RaceCar.__init__ statics      base_classes.py:118-158   -> f110_set_beam_tables
 *   Simulator.update_params       base_classes.py:527-547   -> f110_set_params
 *   Simulator.reset               base_classes.py:627-643   -> f110_sim_reset
 *   Simulator.step + F110Env.step base_classes.py:566-625, f110_env.py:371-421 -> f110_step
 *   F110Env.reset                 f110_env.py:425-472       -> f110_step with reset_mask set
 *
 * Conventions
 *   - N envs x A agents x B beams.  All per-agent arrays are [N][A]..., row-major, env-major.
 *   - Setup calls (create / set_map / set_tables / set_beam_tables / set_params) take HOST
 *     pointers and copy; they synchronise the device.
 *   - f110_step / f110_sim_reset / f110_get_state / f110_set_state take DEVICE pointers into
 *     caller-owned memory (e.g. torch tensors' data_ptr()) and a cudaStream_t passed as void*.
 *     They never allocate and never synchronise: outputs are valid in stream order.
 *   - f110_step_host takes HOST pointers (pinned for full speed), performs the H2D/D2H copies
 *     itself on the handle's stream and returns after synchronising that stream.
 *   - Every call returns F110_OK (0) or a negative F110_ERR_*; f110_last_error() returns a
 *     thread-local message for the last failure.  A handle is bound to one device and must not
 *     be used from two host threads at once.
 *   - There is no CPU fallback: every entry point that computes requires a CUDA device.
 */
#ifndef F110_B200_H
#define F110_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define F110_ABI_VERSION 2

/* vehicle parameter vector, order of the keys of the params dict (f110_env.py:132-156) */
#define F110_NUM_PARAMS 18
enum {
    F110_P_MU = 0, F110_P_C_SF, F110_P_C_SR, F110_P_LF, F110_P_LR, F110_P_H, F110_P_M, F110_P_I,
    F110_P_S_MIN, F110_P_S_MAX, F110_P_SV_MIN, F110_P_SV_MAX, F110_P_V_SWITCH, F110_P_A_MAX,
    F110_P_V_MIN, F110_P_V_MAX, F110_P_WIDTH, F110_P_LENGTH
};

/* Integrator enum values (base_classes.py:40-42) */
#define F110_INTEGRATOR_RK4 1
#define F110_INTEGRATOR_EULER 2

#define F110_MAX_AGENTS 16

enum {
    F110_OK = 0,
    F110_ERR_INVALID = -1,       /* bad argument */
    F110_ERR_MAP_NOT_SET = -2,   /* ValueError('Map is not set for scan simulator.') laser_models.py:445-446 */
    F110_ERR_CUDA = -3,          /* CUDA runtime failure (message in f110_last_error) */
    F110_ERR_INDEX = -4,         /* IndexError('Index given is out of bounds ...') base_classes.py:547 */
    F110_ERR_POSE_COUNT = -5,    /* ValueError('Number of poses for reset ...') base_classes.py:638-639 */
    F110_ERR_INTEGRATOR = -6,    /* SyntaxError('Invalid Integrator Specified ...') base_classes.py:399 */
    F110_ERR_NO_DEVICE = -7      /* no CUDA device: there is no CPU fallback */
};

/* flags for F110Config.flags */
#define F110_FLAG_COUNT_LOOKUPS 1u /* count distance-transform lookups (for the roofline's L-bar) */
#define F110_FLAG_NARROW_FRACTION 2u /* test hook: 6 fraction bits in the lidar kernel's fixed-point cell index, so that
                                        3 % of lookups (instead of 1e-6) finish their ray on the exact-arithmetic path */

typedef struct F110Sim F110Sim;

typedef struct F110Config {
    int32_t abi_version;   /* F110_ABI_VERSION */
    int32_t device;        /* CUDA device ordinal */
    int32_t num_envs;      /* N */
    int32_t num_agents;    /* A  (F110Env kwarg num_agents, f110_env.py:159-162) */
    int32_t num_beams;     /* B  (RaceCar default 1080, base_classes.py:69) */
    int32_t theta_dis;     /* 2000 (laser_models.py:360) */
    int32_t integrator;    /* F110_INTEGRATOR_* (f110_env.py:176-179) */
    int32_t ego_idx;       /* f110_env.py:170-173 */
    uint32_t flags;
    uint32_t host_stream_rank; /* 0: default priority for the f110_step_host* stream; r > 0: r-th highest priority */
    double fov;            /* 4.7 rad (base_classes.py:69) */
    double eps;            /* 1e-4 ray-march termination (laser_models.py:360) */
    double max_range;      /* 30.0 m (laser_models.py:360) */
    double timestep;       /* 0.01 s (f110_env.py:164-167) */
    double lidar_dist;     /* 0.0 (f110_env.py:182-185) */
    double ttc_thresh;     /* 0.005 s (base_classes.py:115) */
    double lidar_max;      /* params['lidar_max'] = 30.0, observation normalisation (f110_env.py:203,559-560) */
    double noise_std;      /* 0.01 m, used only when F110StepIO.noise == NULL (laser_models.py:429) */
    uint64_t seed;         /* seed of the on-device Philox noise stream */
} F110Config;

/* F110StepIO.host_flags: the caller states that host buffers lying exactly back to back were carved out of ONE pinned
 * allocation, so that one copy may span them (see f110_step_host_async).  Without it every field is copied by itself. */
#define F110_HOST_MERGE_ADJACENT 1

/* One step over the whole batch.  Inputs may be NULL where noted; NULL outputs are skipped. */
typedef struct F110StepIO {
    /* ---- inputs */
    const void* actions;         /* [N][A][2] (steer, speed); f32 or f64, see actions_f64.  NULL = zero action */
    int32_t actions_f64;         /* 0: float (train_ddpg.py:171), 1: double (gym_bridge.py:226-228) */
    int32_t host_flags;          /* host path only (f110_step_host*): F110_HOST_MERGE_ADJACENT or 0 */
    const double* noise;         /* [N][A][B] additive lidar noise drawn by the caller (parity mode: numpy's
                                    Generator.normal stream, laser_models.py:450-452); NULL = on-device
                                    Philox2x32-10 + Box-Muller N(0, noise_std^2) */
    const uint8_t* reset_mask;   /* [N] or NULL.  Non-zero: F110Env.reset(options=reset_poses[env]) is applied to the
                                    env first and this step is its zero-action step (f110_env.py:438-458); the env's
                                    action is ignored.  May alias `terminated` (auto-reset on the step after done). */
    const double* reset_poses;   /* [N][A][3] (x, y, yaw); required when reset_mask != NULL */
    const uint8_t* active_mask;  /* [N] or NULL (= all).  Zero: the env is left untouched, outputs not written */
    /* ---- outputs */
    float* obs;                  /* [N][B+8]  F110Env._pack_flat_obs (f110_env.py:552-584) */
    float* reward;               /* [N]       = timestep (f110_env.py:405) */
    uint8_t* terminated;         /* [N]       _check_done (f110_env.py:350) */
    double* scans_f64;           /* [N][A][B] obs-dict scans: noisy, after opponent ray-cast (base_classes.py:617) */
    float* scans_f32;            /* [N][A][B] info['scans'] (f110_env.py:599) */
    double* state;               /* [N][A][7] x, y, steer, v, yaw, yaw_rate, slip after the step (base_classes.py:97) */
    uint8_t* collisions;         /* [N][A]    GJK | iTTC (base_classes.py:563,601-602) */
    int32_t* toggles;            /* [N][A]    toggle_list (f110_env.py:339-346) */
    double* lap_times;           /* [N][A] */
    double* lap_counts;          /* [N][A] */
    double* time;                /* [N]       current_time (f110_env.py:406) */
    double* agent_poses;         /* [N][A][3] Simulator.agent_poses: x, y, yaw after the dynamics update and BEFORE the iTTC
                                    zeroing of a colliding car's yaw (base_classes.py:587 vs :248-250) */
} F110StepIO;

const char* f110_last_error(void);
int f110_abi_version(void);

/* params: F110_NUM_PARAMS doubles applied to every agent (Simulator.__init__, base_classes.py:504-510).
 * Environment switches read here (development / test aids, none changes a result):
 *   F110_DEBUG_SYNC=1   synchronise after every kernel of a step and name the one that faulted
 *   F110_LIDAR_HOMES=n  the lidar kernel's units are cut into n home segments with a queue each, in natural order, instead
 *                       of one per SM for launches above 48 units per resident warp and one below (n is clamped to
 *                       [1, units]; changes the order units run in, never a result)
 * and by f110_set_map_image:
 *   F110_EDT_WIDE=1     force the general form of the device EDT on a map the 16-bit form would take */
int f110_create(const F110Config* cfg, const double* params, F110Sim** out);
void f110_destroy(F110Sim* sim);

/* dt: HOST [height][width] fp64 = resolution * EDT(binarised, bottom-up image) exactly as
 * laser_models.py:398-425 builds it; orig_cos/orig_sin = cos/sin(origin yaw) as computed by the host. */
int f110_set_map(F110Sim* sim, const double* dt, int32_t height, int32_t width, double resolution,
                 double orig_x, double orig_y, double orig_cos, double orig_sin);
/* The same from the binarised image itself: free_mask HOST uint8 [height][width], non-zero = free (pixel > 128), row 0 =
 * bottom image row (laser_models.py:398-404).  The exact Euclidean distance transform (scipy's, laser_models.py:52) runs on
 * the device in integers; the resulting fp64 map is bit-identical to resolution * distance_transform_edt(img). */
int f110_set_map_image(F110Sim* sim, const uint8_t* free_mask, int32_t height, int32_t width, double resolution,
                       double orig_x, double orig_y, double orig_cos, double orig_sin);
/* Device time of the EDT kernels of the last f110_set_map_image call on this handle, in ms (CUDA events); 0 before any. */
float f110_edt_kernel_ms(const F110Sim* sim);
/* Reads the handle's fp64 map back into dt_host (capacity in cells).  On a map set: slot 0's map. */
int f110_get_map(F110Sim* sim, double* dt_host, int64_t capacity_cells);

/* ---- map sets: several maps in one handle, each env driving on the map of its SLOT (DESIGN.md section 10) ----
 * Every env's dynamics, lidar, iTTC, collisions and observation are exactly what a handle holding only that env's map would
 * produce, bit for bit.  All maps of a set are padded to ONE fixed-point format, the one the largest side in the set gets
 * alone (see f110_set_map), and lie back to back in one allocation: each member costs as much device memory as the largest
 * would.  A set that contains one 8000 x 8000 map pads every member to 8208 x 8192 cells = 538 MB.  The set's padded cells
 * in all must stay below 2^31 (31 maps when the largest is 8000^2, 127 at 4000^2, 508 at 2000^2).
 * The shaped reward (f110_reward_*) keeps one centerline per reward object: it does not know about slots. */
#define F110_MAX_MAPS 256
typedef struct F110MapDesc {
    const double*  dt;         /* HOST [height][width] fp64 as f110_set_map takes it, or NULL */
    const uint8_t* free_mask;  /* HOST [height][width] as f110_set_map_image takes it; used when dt == NULL (device EDT) */
    int32_t height, width;
    double resolution, orig_x, orig_y, orig_cos, orig_sin;
} F110MapDesc;
/* Installs `count` (1 .. F110_MAX_MAPS) maps at once; maps may differ in size, resolution and origin.  Afterwards env e
 * drives on slot floor(e * count / N) (contiguous blocks, which keep the lidar kernel's home-segment locality).  Atomic: on
 * any failure (F110_ERR_INVALID for bad arguments or a set too large, F110_ERR_CUDA for out of memory) the handle keeps
 * the map or maps it had.  Bumps f110_map_generation.  A set of one map is f110_set_map / f110_set_map_image of that map,
 * and f110_set_map / f110_set_map_image on a handle holding a set replace the set with that one map. */
int f110_set_maps(F110Sim* sim, const F110MapDesc* maps, int32_t count);
/* Maps installed: 1 for a single map, 0 before any. */
int32_t f110_map_count(const F110Sim* sim);
/* Reads map `slot` back like f110_get_map; slot outside [0, f110_map_count) -> F110_ERR_INDEX. */
int f110_get_map_slot(F110Sim* sim, int32_t slot, double* dt_host, int64_t capacity_cells);
/* Slot assignment, stream-ordered (capturable into a CUDA graph; does NOT bump f110_map_generation).  slots DEVICE int32
 * [N], env_mask DEVICE uint8 [N] or NULL (= all); entries outside [0, count) leave that env's slot unchanged.  An env whose
 * slot changes without a reset goes on from the same coordinates on the other map (as the reference's update_map does);
 * reset it in the same step to start it anew.  The assignment is not part of the f110_get_state blob. */
int f110_set_env_maps(F110Sim* sim, const int32_t* slots, const uint8_t* env_mask, void* stream);
/* The same from HOST arrays: validates first (an entry out of range -> F110_ERR_INDEX, nothing changed), copies, synchronises. */
int f110_set_env_maps_host(F110Sim* sim, const int32_t* slots, const uint8_t* env_mask);
/* slots_out: DEVICE int32 [N] <- each env's slot, stream-ordered. */
int f110_get_env_maps(F110Sim* sim, int32_t* slots_out, void* stream);
/* HOST [theta_dis] tables (laser_models.py:379-381). */
int f110_set_tables(F110Sim* sim, const double* sines, const double* cosines);
/* HOST [B] tables (base_classes.py:125-158).  scan_angles must be strictly increasing. */
int f110_set_beam_tables(F110Sim* sim, const double* scan_angles, const double* beam_cosines,
                         const double* side_distances);
/* agent_idx < 0: all agents; otherwise that agent in every env; >= A -> F110_ERR_INDEX. */
int f110_set_params(F110Sim* sim, const double* params, int32_t agent_idx);

/* Simulator.reset: poses DEVICE [N][A][3]; num_poses must equal A (else F110_ERR_POSE_COUNT);
 * env_mask DEVICE [N] or NULL.  Does not step. */
int f110_sim_reset(F110Sim* sim, const double* poses, int32_t num_poses, const uint8_t* env_mask, void* stream);
/* The same with HOST pointers: copies, resets on the internal stream and synchronises it (for callers without device
 * memory of their own, e.g. the ctypes Simulator of INTEGRATION.md). */
int f110_sim_reset_host(F110Sim* sim, const double* poses, int32_t num_poses, const uint8_t* env_mask);

int f110_step(F110Sim* sim, const F110StepIO* io, void* stream);

/* Same contract with HOST pointers in `io`; copies in and out on an internal stream and synchronises it. */
int f110_step_host(F110Sim* sim, const F110StepIO* io);
/* The same without the final synchronisation: the host buffers are valid after f110_host_sync().  Lets a caller
 * that shards its envs over several handles overlap one shard's PCIe copies with another shard's kernels.
 * With F110_HOST_MERGE_ADJACENT in io->host_flags, fields whose host buffers lie exactly back to back in the order
 *     inputs : actions, reset_poses, noise, reset_mask, active_mask
 *     outputs: scans_f64, state, lap_times, lap_counts, time, obs, scans_f32, reward, toggles, terminated, collisions
 * (absent fields skipped) are moved by a single copy per direction; fields placed otherwise get one copy each. */
int f110_step_host_async(F110Sim* sim, const F110StepIO* io);
int f110_host_sync(F110Sim* sim);
/* f110_step_host_async on `count` handles (ios[i] belongs to sims[i]), then f110_host_sync on each: one call per step
 * for a caller that shards its envs over several handles. */
int f110_step_host_multi(F110Sim* const* sims, const F110StepIO* ios, int32_t count);

/* Checkpoint of the whole persistent simulation state as one opaque blob (DEVICE pointer): a 64-byte header (magic, layout
 * version, N, A, B, size) followed by the state arena.  f110_set_state reads the header back (it synchronises the stream)
 * and refuses a blob of another layout version or batch shape with F110_ERR_INVALID.  What the blob does NOT hold is the
 * caller's: the terminated flags it uses as the next reset mask, its start poses, host-side noise generators --
 * F110VecEnv.state_dict / F110Env.state_dict add those. */
int64_t f110_state_nbytes(const F110Sim* sim);
int f110_get_state(F110Sim* sim, void* dst, void* stream);
int f110_set_state(F110Sim* sim, const void* src, void* stream);

/* Episode statistics accumulated on the device since the last call with reset != 0.
 * out: DEVICE double[F110_NUM_STATS]; meant to be all-reduced (sum) across ranks off the step path. */
#define F110_NUM_STATS 8
enum { F110_STAT_EPISODES = 0, F110_STAT_EPISODE_STEPS, F110_STAT_EGO_COLLISIONS, F110_STAT_LAPS_DONE,
       F110_STAT_EPISODE_TIME, F110_STAT_RESERVED5, F110_STAT_RESERVED6, F110_STAT_RESERVED7 };
int f110_get_stats(F110Sim* sim, double* out, int32_t reset, void* stream);

/* Sum of distance-transform lookups since creation (requires F110_FLAG_COUNT_LOOKUPS); synchronises. */
int f110_get_lookup_count(F110Sim* sim, uint64_t* lookups, uint64_t* rays);
/* Longest ray (in lookups) seen so far, as of the last f110_get_lookup_count call. */
int64_t f110_max_lookups(const F110Sim* sim);
/* Rays the lidar kernel redid in the reference's own arithmetic because its fixed-point march met a lookup it could not
 * decide (cell-edge guard band, map border and beyond, non-finite pose), as of the last f110_get_lookup_count call. */
int64_t f110_redone_rays(const F110Sim* sim);
/* The lidar kernel variant the last step selected (host-side record, no synchronisation): out[0] the fraction bits of
 * the map (of the set's common format), out[1] the template fraction bits (19..22 for a tuned variant, 0 for the generic
 * one), out[2] the mode (0 opponents, 1 single agent, 2 single agent lean, 3 opponents lean), out[3] 1 when a map
 * set's kernel ran.  F110_ERR_INVALID before the first step. */
int f110_get_lidar_variant(const F110Sim* sim, int32_t out[4]);
/* Development aid (requires F110_FLAG_COUNT_LOOKUPS): per work unit of the last lidar launch, 4 words (start ns, end ns,
 * both the low half of %globaltimer; longest ray in lookups | lanes redone exactly << 24; sm << 24 | queue position).  out == NULL returns the number
 * of units (0 when no timeline is kept); otherwise copies [units][4] words and returns the count, or a negative error. */
int64_t f110_debug_unit_timeline(F110Sim* sim, uint32_t* out, int64_t capacity_units);
/* Incremented by every successful f110_set_map / f110_set_map_image / f110_set_maps (not by f110_set_env_maps).  The step kernels receive the map descriptor by
 * value, so a CUDA graph captured from f110_step before a map change still holds the old (freed) map: re-capture when
 * this number has changed (F110VecEnv does). */
int64_t f110_map_generation(const F110Sim* sim);

/* Per-kernel timing for bench.py's roofline: when enabled every f110_step records CUDA events around its three
 * kernels on the launch stream (not capturable into a CUDA graph while enabled).  f110_get_kernel_timing
 * synchronises, writes the summed milliseconds of {dynamics, lidar, post} and the number of steps, and clears. */
int f110_set_kernel_timing(F110Sim* sim, int32_t enable);
int f110_get_kernel_timing(F110Sim* sim, double* ms3, int64_t* steps);

/* Launch bookkeeping for bench.py: kernels launched by this handle since creation. */
int64_t f110_kernel_launches(const F110Sim* sim);

/* ---- consumers around the env, on the device (SURVEY 8f) ----
 * gap_follow_action (rl_training/utils/gap_follow.py:43-58), the rule-based opponent train_ddpg.py:168 drives from
 * info["scans"][1]: for scan k (DEVICE float[num_beams] at scans + k*scan_stride) writes (steer, speed) as two floats
 * at actions + k*action_stride.  Defaults of the reference: angle_min = -pi/2, angle_increment = pi/1080,
 * max_distance 3.0, window_size 5, bubble_radius 30, threshold 0.5.  Strides are in elements. */
int f110_gap_follow(const float* scans, int64_t num_scans, int64_t scan_stride, int32_t num_beams,
                    float* actions, int64_t action_stride, double angle_min, double angle_increment,
                    float max_distance, int32_t window_size, int32_t bubble_radius, float threshold, void* stream);

/* CenterlineSafetyProgressReward (rl_training/utils/rewards.py:185-355) over CenterlineProgress
 * (rl_training/utils/track_progress.py), the reward train_ddpg.py:127-145,179 computes from the flat observation; one
 * independent reward object (progress tracker state included) per env.  Field names and defaults are the constructor's. */
typedef struct F110RewardConfig {
    int32_t num_envs, num_points, num_beams, device;
    int32_t closed;             /* CenterlineProgress(closed=True) */
    int32_t grace_steps_wall, grace_steps_opp, reserved;
    double dt, w_prog, forward_sign, alive_bonus, w_rel_lead, lead_clip, w_lat, lat_cap, default_half_width, lidar_max,
           near_wall_dist, w_wall, wall_quantile, opp_safe_dist, w_opp, ego_crash_penalty, opp_crash_bonus;
} F110RewardConfig;
typedef struct F110Reward F110Reward;
/* xy: HOST [num_points][2] centerline, 2 <= num_points <= 16385; wR / wL: HOST [num_points] half-widths or NULL (CSV columns w_tr_right_m / _left_m). */
int f110_reward_create(const F110RewardConfig* cfg, const double* xy, const double* wR, const double* wL, F110Reward** out);
void f110_reward_destroy(F110Reward* r);
/* obs: DEVICE float [num_envs][num_beams + 8] (F110StepIO.obs); reset_mask: DEVICE [num_envs] or NULL, non-zero =
 * reward_fn.reset() before this call; out_f64 / out_f32: DEVICE [num_envs], either may be NULL. */
int f110_reward_compute(F110Reward* r, const float* obs, const uint8_t* reset_mask, double* out_f64, float* out_f32, void* stream);

/* ---- measurement utility: the empirical dependent-gather roofline (SURVEY 8d) ----
 * num_threads threads each chase `chain` dependent 8-byte loads through a power-of-two window of `window_cells`
 * (<= 0: the whole map) cells of the DEVICE fp64 array map_dev; ms_out receives the average kernel time over
 * `repeats` launches.  Synchronises. */
int f110_gather_probe(const double* map_dev, int64_t num_cells, int64_t window_cells, int32_t chain,
                      int64_t num_threads, int32_t repeats, double* sink_dev, float* ms_out, void* stream);

/* ---- development aid: the dynamics kernel's trig, compiled with the library's flags ----
 * For each DEVICE x_dev[i], i < n, writes into the DEVICE array out_dev [4][n]: out[0][i], out[1][i] = sin, cos from one
 * sincos(x) call (the heading terms), out[2][i] = tan(x), out[3][i] = cos(x) (the steering angle of the kinematic
 * branch).  A model of the dynamics kernel that takes its trig from here reproduces the kernel bit for bit.  Enqueues on
 * `stream`, does not synchronise. */
int f110_trig_probe(const double* x_dev, int64_t n, double* out_dev, void* stream);
/* The shaped reward's hypot, compiled with the library's flags: out_dev[i] = hypot(a_dev[i], b_dev[i]) for i < n, all
 * DEVICE arrays.  With f110_trig_probe's sincos it is all a model of the reward kernels needs beyond IEEE arithmetic to
 * reproduce them bit for bit.  Enqueues on `stream`, does not synchronise. */
int f110_hypot_probe(const double* a_dev, const double* b_dev, int64_t n, double* out_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* F110_B200_H */
