/*
 * jss_b200.h -- C-ABI of the B200-native batched job-shop environment.
 *
 * The reference (prosysscience/JSSEnv) has NO FFI layer: its boundary is the
 * Python object protocol of `JssEnv` (JSSEnv/envs/jss_env.py:14).  Each entry
 * point below names the reference interface it replaces (file:line relative to
 * the reference tree).  The Python mirror of that interface lives in
 * jssenv_b200/ (JssEnv / JssVecEnv / dispatching) and binds these symbols with
 * ctypes; INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions
 *   - plain pointers and sizes only; no C++/torch types cross this boundary;
 *   - every call returns JSS_OK (0) or a negative JSS_ERR_* code and never throws;
 *     jss_last_error() gives the message for the handle (or for creation if NULL);
 *   - the library owns all device memory; jss_get_buffers() exposes device
 *     pointers that stay valid until jss_destroy(); callers wrap them zero-copy;
 *   - all work is enqueued on the `stream` argument (a cudaStream_t passed as
 *     void*; NULL = the legacy default stream) and is asynchronous unless the
 *     call says otherwise; a handle is bound to ONE device and is not thread-safe
 *     (multi-GPU = one process/handle per GPU);
 *   - there is NO CPU fallback: without a CUDA device jss_create() fails with
 *     JSS_ERR_NO_DEVICE.
 *
 * Batched semantics (N independent envs; env i runs instance env_to_inst[i]):
 *   action a in [0, J_i)  allocate job a            (jss_env.py:441-481)
 *   action a == J_i       no-op / wait              (jss_env.py:419-440)
 *   action JSS_ACTION_SKIP     leave env i untouched this call
 *   action JSS_ACTION_ADVANCE  raw increase_time_step() (jss_env.py:495-637),
 *                              the hook tests/test_solutions.py:66 calls directly
 *   Reference exceptions become a per-env sticky error bit (JSS_FLAG_ERROR) and
 *   the env is left unchanged for that call: job action that is not legal,
 *   finished job (IndexError jss_env.py:444), no-op with no pending event
 *   (IndexError jss_env.py:517), out-of-range action.
 *   A done env is frozen (its terminal observation stays readable) until it is
 *   reset; with JSS_CREATE_AUTO_RESET the next jss_step() on it performs the
 *   reset instead (reward 0, done 0).
 */
#ifndef JSS_B200_H
#define JSS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define JSS_ABI_VERSION 3

/* limits of the one-warp-per-env kernels */
#define JSS_MAX_JOBS 256
#define JSS_MAX_MACHINES 32
#define JSS_MAX_DURATION 2047

/* return codes */
#define JSS_OK 0
#define JSS_ERR_INVALID (-1)     /* bad argument */
#define JSS_ERR_NO_DEVICE (-2)   /* no CUDA device / wrong architecture */
#define JSS_ERR_CUDA (-3)        /* a CUDA runtime call failed (see jss_last_error) */
#define JSS_ERR_UNSUPPORTED (-4) /* instance exceeds JSS_MAX_*, or has a zero-length op (the reference cannot finish such an
                                    episode either: jss_env.py:529 never sees the op as completed) */
#define JSS_ERR_STATE (-5)       /* call order violated (e.g. step before load/assign) */

/* special actions */
#define JSS_ACTION_SKIP (-1)
#define JSS_ACTION_ADVANCE (-2)

/* jss_create flags */
#define JSS_CREATE_AUTO_RESET 1u      /* step() on a done env resets it */
#define JSS_CREATE_RECORD_SOLUTION 2u /* keep solution[N][Jmax][Mmax] start times (jss_env.py:163,454) */
#define JSS_CREATE_HOST_MIRROR 4u     /* small batches (the single-env facade): action_mask, real_obs, the scalar records,
                                         the x_* arrays and an action slot live in ONE pinned, device-mapped host block --
                                         the kernels write results straight into host memory, no copies per transition */

/* per-env flag bits (jss_buffers.flags_done >> 8) */
#define JSS_FLAG_DONE 1u        /* _is_done() (jss_env.py:639-653) */
#define JSS_FLAG_ERROR 2u       /* sticky until reset */
#define JSS_FLAG_NOOP_LEGAL 4u  /* legal_actions[J] */

/* dispatching rules (JSSEnv/dispatching.py); RANDOM = masked-uniform policy
 * (README.md:58-60) */
#define JSS_RULE_RANDOM 0
#define JSS_RULE_SPT 1   /* dispatching.py:92-116  */
#define JSS_RULE_FIFO 2  /* dispatching.py:133-156 */
#define JSS_RULE_MWR 3   /* dispatching.py:173-199 */
#define JSS_RULE_LWR 4   /* dispatching.py:216-242 */
#define JSS_RULE_MOR 5   /* dispatching.py:259-283 */
#define JSS_RULE_LOR 6   /* dispatching.py:300-324 */
#define JSS_RULE_CR 7    /* dispatching.py:365-408 */
#define JSS_NUM_RULES 8

/* jss_policy coin modes for the rules' "10 % wait" draw (dispatching.py:113) */
#define JSS_COIN_DEVICE 0 /* counter RNG: wait iff hash(seed, env, step) < 0.1 * 2^32 */
#define JSS_COIN_NEVER 1  /* never wait; caller reads JSS_FLAG_NOOP_LEGAL and decides (host np.random) */

typedef struct jss_handle jss_t;

/* Device pointers owned by the library (jss_get_buffers).
 * Layout: row-major, env-major.  J = jobs_max, M = machines_max of the batch. */
typedef struct jss_buffers {
    int32_t n_envs;
    int32_t jobs_max;       /* J */
    int32_t machines_max;   /* M */
    int32_t mask_stride;    /* bytes per action_mask row (>= J+1, multiple of 4) */
    uint8_t *action_mask;   /* [N][mask_stride]; bytes 0..J_i = legal_actions of env i (jss_env.py:133) */
    float *real_obs;        /* [N][J][7] fp32 (jss_env.py:102-111, 132)            */
    int32_t scalar_stride;  /* bytes between consecutive envs in the five per-env scalar arrays below
                               (they are fields of one 16-byte record per env, written with one store) */
    int32_t host_mirror;    /* 1: the output pointers below are host-readable (JSS_CREATE_HOST_MIRROR) */
    float *reward;          /* [N] scaled reward (jss_env.py:483-493)              */
    int32_t *reward_raw;    /* [N] reward before scaling; -hole for ACTION_ADVANCE */
    uint8_t *done;          /* [N] 0/1 (low byte of flags_done)                    */
    int32_t *time;          /* [N] current_time_step (makespan once done)          */
    uint32_t *flags_done;   /* [N] (JSS_FLAG_* << 8) | done                        */
    int32_t *solution;      /* [N][J][M] or NULL (JSS_CREATE_RECORD_SOLUTION)      */
    /* per-env episode statistics, updated when an episode ends */
    int32_t *episode_count;     /* [N] finished episodes               */
    int32_t *last_makespan;     /* [N] makespan of the last finished episode (jss_env.py:650) */
    int32_t *last_return;       /* [N] raw return of the last finished episode */
    /* canonical (decoded) state, filled by jss_export_state only */
    int32_t *x_todo;        /* [N][J] todo_time_step_job                  */
    int32_t *x_tufco;       /* [N][J] time_until_finish_current_op_jobs   */
    int32_t *x_idle_last;   /* [N][J] idle_time_jobs_last_op              */
    int32_t *x_total_idle;  /* [N][J] total_idle_time_jobs                */
    int32_t *x_col4;        /* [N][J] numerator of real_obs[:,4]; max_time_op encodes 1.0 */
    int32_t *x_tuam;        /* [N][M] time_until_available_machine        */
    uint8_t *x_legal;       /* [N][J] legal_actions[:-1]                  */
    uint8_t *x_blocked;     /* [N][J] action_illegal_no_op                */
    int32_t *mirror_actions; /* [N] action slot inside the host block (JSS_CREATE_HOST_MIRROR), else NULL */
} jss_buffers;

/* number of int64 slots jss_stats() writes */
#define JSS_STATS_LEN 8
/* [0] finished episodes  [1] env steps executed  [2] sum of makespans
 * [3] min makespan (INT64_MAX if none)  [4] max makespan  [5] sum of raw returns
 * [6] envs currently done  [7] envs with the error bit set */

/* --- lifetime ---------------------------------------------------------- */

/* Replaces JssEnv.__init__ (jss_env.py:27-119) for a batch of n_envs envs on CUDA
 * device `device`.  `env_id_base` is the global index of env 0 (multi-GPU
 * shards: rank r passes r * n_envs so RNG streams do not depend on the world
 * size). */
int jss_create(jss_t **out, int device, int n_envs, uint32_t flags, uint64_t env_id_base);
void jss_destroy(jss_t *h);
const char *jss_last_error(const jss_t *h);
int jss_abi_version(void);

/* Replaces the instance parse (jss_env.py:72-95): n_inst instances, instance k
 * has jobs[k] x machines[k] operations stored row-major at
 * machine[offsets[k] ...] / duration[offsets[k] ...] (host pointers). */
int jss_load_instances(jss_t *h, int n_inst, const int32_t *jobs, const int32_t *machines,
                       const int64_t *offsets, const int32_t *machine, const int32_t *duration);

/* env i runs instance env_to_inst[i] (host pointer, n_envs entries); allocates
 * all device buffers.  Must follow jss_load_instances. */
int jss_assign(jss_t *h, const int32_t *env_to_inst);

int jss_get_buffers(jss_t *h, jss_buffers *out);

/* derived per-instance scalars (jss_env.py:86-89): out[0]=max_time_op,
 * out[1]=max_time_jobs, out[2]=sum_op */
int jss_instance_scalars(jss_t *h, int inst, int64_t out[3]);

/* --- generator mode: a fresh random instance per env and episode ------------------------------------------
 * Instance k of global env g (env_id_base + i) under instance seed s, for shape J x M and durations in
 * [dmin, dmax], is a pure function of those values, computed with the same integer code on host and device
 * (jssenv_b200/csrc/jss_gen.h):
 *   h(c)            = jss_hash3(s ^ 0x6A09E667F3BCC909, g, c)     (the policy RNG uses jss_hash3(seed, g, step))
 *   c(j, i, w)      = (k << 20) | (((j * M + i) << 1) | w)
 *   duration[j][i]  = dmin + pick(h(c(j, i, 0)), dmax - dmin + 1)
 *   machine[j]      = Fisher-Yates shuffle of 0..M-1 (Taillard): from the identity, for i = 0 .. M-2,
 *                     r = i + pick(h(c(j, i, 1)), M - i), swap positions i and r;
 *   pick(x, n)      = (x * n) >> 32 (64-bit product), jss_hash3 as in jssenv_b200/csrc/jss_rng.h.
 * k counts the resets of the env: 0 at the reset jss_assign_generated performs, +1 at every later reset, explicit
 * (jss_reset, masked or not) or automatic.  The stream does not depend on sharding; a second handle with the same
 * seed replays it.  Limits: 2 <= M <= 32, 1 <= J <= 128, 1 <= dmin <= dmax <= 2047; all envs share one shape.
 * In this mode jss_import_state, jss_step_export, jss_instance_scalars and the packed / hybrid host steps return
 * JSS_ERR_UNSUPPORTED; everything else works as for loaded instances. */

/* Takes the place of jss_load_instances + jss_assign on a fresh handle: allocates per-env instance tables,
 * draws instance 0 of every env on the device and resets.  JSS_ERR_STATE after either of the two,
 * JSS_ERR_UNSUPPORTED with JSS_CREATE_HOST_MIRROR. */
int jss_assign_generated(jss_t *h, int jobs, int machines, int dur_min, int dur_max, uint64_t inst_seed);

/* Each env's current instance: machine_dev / duration_dev int32 [N][J][M], index_dev int32 [N] (its k).
 * Device pointers, any may be NULL; enqueued on `stream`. */
int jss_get_env_instances(jss_t *h, int32_t *machine_dev, int32_t *duration_dev, int32_t *index_dev, void *stream);

/* Host restatement of the generator (no device needed): instance `index` of env `env_id` into
 * machine_host / duration_host int32 [J][M]. */
int jss_generate_instance(int jobs, int machines, int dur_min, int dur_max, uint64_t inst_seed, uint64_t env_id,
                          uint64_t index, int32_t *machine_host, int32_t *duration_host);

/* --- hot path ------------------------------------------------------------ */

/* Replaces reset() (jss_env.py:145-181).  env_mask_dev: device u8[N], nonzero =
 * reset that env; NULL = reset all. */
int jss_reset(jss_t *h, const uint8_t *env_mask_dev, void *stream);

/* Replaces step() (jss_env.py:403-481) incl. increase_time_step (495-637),
 * _prioritization_non_final (183-254), _check_no_op (256-401), _reward_scaler
 * (483-493), _is_done (639-653), _get_current_state_representation (121-134).
 * actions_dev: device int32[N]. */
int jss_step(jss_t *h, const int32_t *actions_dev, void *stream);

/* jss_step() + jss_export_state() in ONE launch (generic kernel): the latency path of the single-env facade, which
 * needs the decoded state after every transition to serve the reference's attribute surface. */
int jss_step_export(jss_t *h, const int32_t *actions_dev, void *stream);

/* Replaces DispatchingRule.__call__ (dispatching.py:92-408) / the masked-random
 * sampler (README.md:58-60).  Writes device int32[N] actions.  `step_index` is
 * the RNG counter (callers increment it per decision). */
int jss_policy(jss_t *h, int rule, int coin_mode, uint64_t seed, uint64_t step_index,
               int32_t *actions_dev, void *stream);

/* Replaces CriticalRatio.__init__(due_date_factor) (dispatching.py:337-349): the factor JSS_RULE_CR multiplies a
 * job's total processing time with to get its due date (dispatching.py:357-360).  Default 1.5 like the reference;
 * applies to every later jss_policy / jss_step_sample / jss_rollout with JSS_RULE_CR on this handle. */
int jss_set_cr_due_date_factor(jss_t *h, double factor);

/* jss_step() fused with jss_policy() for the NEXT decision: applies actions_dev, then
 * writes every env's next action (chosen by `rule` on the new state, RNG counter
 * `step_index`) to next_actions_dev, in one launch.  The two buffers may alias. */
int jss_step_sample(jss_t *h, const int32_t *actions_dev, int rule, int coin_mode, uint64_t seed,
                    uint64_t step_index, int32_t *next_actions_dev, void *stream);

/* Replaces DispatchingRule.run_episode (dispatching.py:55-75) for the whole
 * batch: n_steps x (policy -> step) fused in one launch, state kept on chip
 * between steps; observations are written every step iff write_obs != 0. */
int jss_rollout(jss_t *h, int rule, uint64_t seed, uint64_t step_index, int n_steps,
                int write_obs, void *stream);

/* jss_rollout() that also RECORDS the trajectory (what an on-policy collector wants from a rule / random policy):
 * for k < n_steps and env e, slot k * N + e of the caller's device buffers receives the outputs of transition k --
 * traj_obs [n_steps][N][J][7] fp32, traj_mask [n_steps][N][mask_stride] u8, traj_scalars [n_steps][N][4] int32
 * (the 16-byte records), traj_actions [n_steps][N] int32 (the action taken; may be NULL).  The regular buffers hold
 * the last transition afterwards, as after jss_rollout.  n_steps * N < 2^31. */
int jss_rollout_traj(jss_t *h, int rule, uint64_t seed, uint64_t step_index, int n_steps, float *traj_obs,
                     uint8_t *traj_mask, int32_t *traj_scalars, int32_t *traj_actions, void *stream);

/* Host-buffer form of step(): copies actions H2D, steps, copies the results D2H with
 * contiguous DMA, synchronises.  Any output pointer may be NULL.  Host layouts equal the
 * device layouts: mask_host [N][mask_stride] bytes (row i: bytes 0..J_i), obs_host
 * [N][J][7] fp32, scalars_host [N][4] int32 = the 16-byte records
 * {reward (fp32 bits), reward_raw, current_time_step, flags << 8 | done}. */
int jss_step_host(jss_t *h, const int32_t *actions_host, uint8_t *mask_host, float *obs_host,
                  int32_t *scalars_host, void *stream);

/* Pipelined host-buffer stepping (the e2e path).  jss_host_step_begin enqueues, on internal
 * streams, H2D of the actions, the step kernel, D2H of mask + scalar records (small, first) and
 * the D2H of real_obs via a device staging copy, and returns immediately.
 * jss_host_wait(JSS_WAIT_MASK) blocks until mask/scalars of the latest begin have landed (enough
 * for a host policy to choose the next actions); JSS_WAIT_OBS until its observation has landed.
 * A new begin may follow WAIT_MASK while the previous observation is still streaming into ITS host
 * buffer (callers alternate two pinned observation buffers and call WAIT_OBS before reading one).
 * The pipeline is ordered after the work already enqueued on `after_stream` (the caller's stream);
 * call jss_host_wait(JSS_WAIT_OBS) before going back to the stream-ordered entry points. */
#define JSS_WAIT_MASK 1
#define JSS_WAIT_OBS 2       /* observation of the latest begin */
#define JSS_WAIT_OBS_PREV 3  /* observation of the begin before the latest one */
#define JSS_WAIT_WIRE 4      /* packed rows of the latest begin (they precede its fp32 rows on the copy stream) */
int jss_host_step_begin(jss_t *h, const int32_t *actions_host, uint8_t *mask_host, float *obs_host,
                        int32_t *scalars_host, void *after_stream);
int jss_host_wait(jss_t *h, int what);

/* Packed form of the pipelined host-buffer step: instead of the 28 bytes per job of fp32 real_obs, 10 bytes per job
 * cross PCIe -- the INTEGER numerators of the observation columns (jss_env.py:102-111: legal bit,
 * time_until_finish_current_op, todo_time_step, the stale column-4 numerator, idle_time_jobs_last_op,
 * total_idle_time_jobs; column 3 is derivable) -- and jss_host_expand_obs() rebuilds the exact float observation
 * on the host (multi-threaded; same correctly rounded quotients as the device real_obs, bit for bit).
 * wire_host: [N][jss_host_wire_stride()] bytes (pinned).  scalars_host is required (the expansion reads
 * current_time_step from it).  Waiting works as for jss_host_step_begin: JSS_WAIT_OBS* = the wire rows have landed. */
int jss_host_step_begin_packed(jss_t *h, const int32_t *actions_host, uint8_t *mask_host, uint8_t *wire_host,
                               int32_t *scalars_host, void *after_stream);
/* Hybrid: the first n_dma envs ship their observation as final fp32 rows by DMA (obs_host rows [0, n_dma)), the rest as
 * packed rows (wire_host rows [n_dma, N)) to be expanded with jss_host_expand_obs_range(.., n_dma, N) -- PCIe and the
 * host cores work in parallel, each on its share.  obs_host: pinned [N][J][7] fp32 (also the expansion target). */
int jss_host_step_begin_hybrid(jss_t *h, const int32_t *actions_host, uint8_t *mask_host, uint8_t *wire_host,
                               float *obs_host, int n_dma, int32_t *scalars_host, void *after_stream);
int jss_host_expand_obs_range(jss_t *h, const uint8_t *wire_host, const int32_t *scalars_host, float *obs_host,
                              int env_begin, int env_end);
int64_t jss_host_wire_stride(jss_t *h);
/* wire rows + scalar records of one step -> obs_host [N][J][7] fp32 (rows of env i: J_i * 7 floats written). */
int jss_host_expand_obs(jss_t *h, const uint8_t *wire_host, const int32_t *scalars_host, float *obs_host);

/* Host worker pool shared by jss_host_masked_random / jss_host_expand_obs: `threads` workers (0 = the CPUs this
 * process may use, divided by LOCAL_WORLD_SIZE under torchrun); bind_numa_of_device >= 0 binds them (and the calling
 * thread) to the CPUs of that GPU's NUMA node.  Returns the number of CPUs bound (0 = unbound).  Call before first use. */
int jss_host_configure(int threads, int bind_numa_of_device);
int jss_host_threads(void);
/* Cap the SIMD level of jss_host_expand_obs: 0 scalar, 1 AVX2, 2 AVX-512 (default: best available).  For tests. */
int jss_host_set_simd(int level);

/* --- auxiliary ----------------------------------------------------------- */

/* Per-shard statistics (host int64[JSS_STATS_LEN]); synchronises `stream`. */
int jss_stats(jss_t *h, int64_t *out_host, void *stream);

/* Decode the packed device state into the canonical x_* arrays / load it back
 * (snapshot & restore).  env_mask_dev as in jss_reset. */
int jss_export_state(jss_t *h, void *stream);
int jss_import_state(jss_t *h, const uint8_t *env_mask_dev, void *stream);

/* Host utility with the device policy's RNG: masked-uniform action per env from
 * a host mask of n rows of `width` (= J+1) bytes, `row_stride` bytes apart, for
 * host-side agents and tests (multi-threaded for large batches). */
int jss_host_masked_random(const uint8_t *mask_host, int n, int width, int64_t row_stride, uint64_t seed,
                           uint64_t env_id_base, uint64_t step_index, int32_t *actions_host);

/* Number of kernels this handle has launched so far (bench.py's gpu_launches). */
int64_t jss_launch_count(const jss_t *h);

#ifdef __cplusplus
}
#endif
#endif /* JSS_B200_H */
