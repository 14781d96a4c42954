// Host/device shared plain-data types of the batched job-shop kernels.
#pragma once
#include <stdint.h>

// ---- packed instance tables (read-only, built by jss_load_instances) ----------
// ops_pool  u16 [J*M]      op = (machine << 11) | duration   (M <= 32, duration <= 2047)
// len_pool  i32 [J]        jobs_length[j] = sum of durations (jss_env.py:87)
// rem_pool  u16 [J*(M+1)]  rem[j][k] = sum of durations of ops k..M-1 (rules MWR/LWR/CR)
#define JSS_OP_SHIFT 11
#define JSS_OP_DMASK 2047u
#define JSS_OP_NONE 0xFFFFFFFFu  // register-only marker "job has no current op" (finished / padding): machine field >= 32

struct JssInstDesc {
    int32_t J, M;
    int32_t max_time_op, max_time_jobs, sum_op;  // jss_env.py:86-89
    int32_t ops_off;                              // offsets into the pools, in elements
    int32_t len_off;
    int32_t rem_off;
    // correctly rounded fp32 reciprocals of the four observation divisors (jss_div)
    float r_mto, r_mtj, r_sop, r_M;
};

// ---- per-env state block in HBM (int32 words; every sub-array 16-byte aligned) ---
//   [0      , Jcap )   todo_time_step_job            (padding slots hold M)
//   [Jcap   , 2Jcap)   time_until_finish_current_op_jobs
//   [2Jcap  , 3Jcap)   idle_time_jobs_last_op
//   [3Jcap  , 4Jcap)   total_idle_time_jobs
//   [4Jcap  , 5Jcap)   numerator of real_obs[:,4] (stale by design, jss_env.py:569-586)
//   [5Jcap  , +Mcap)   time_until_available_machine
//   then 8 words  = 32 bytes, byte l = lane l's job bits: bit i legal(job KJ*l+i),
//                   bit 4+i blocked by a no-op (action_illegal_no_op)
//                   (instances with 129..256 jobs, KJ = 8: 16 words, one 16-bit word per lane, blocked = bit 8+i)
//        4 words  header: current_time_step, flags, episode_steps, episode_return_raw
// Jcap / Mcap are those of the ENV'S OWN instance (J, M rounded up to a multiple of 4), not batch maxima.
// Not stored because derivable (SURVEY.md section 8 a13): event queue, illegal_actions
// [M][J], machine_legal, both counters, needed_machine_jobs, total_perform_op_time_jobs.
#define JSS_HDR_T 0
#define JSS_HDR_FLAGS 1
#define JSS_HDR_EP_STEPS 2
#define JSS_HDR_EP_RETURN 3

struct JssTile {       // one CTA work item: up to `count` envs of ONE instance (one 16-byte load)
    int32_t first;     // index into `order`
    int32_t inst_count;  // (instance << 8) | count
    // The state blocks are stored in TILE order with the block size of the env's own instance (a mixed batch
    // moves 432 B for a 15x15 env and 2 128 B for a 100x20 env, not the batch maximum): warp w of this tile
    // owns the block at 16-byte unit  state_off16 + w * block16.
    uint32_t state_off16;
    uint32_t block16;  // block size of this tile's instance in 16-byte units
};

struct JssCtaRange {   // mixed batches: the tiles of one persistent CTA -- an equal slice of EVERY lane class
    int32_t a4, b4, a2, b2;     // [a4, b4) KJ = 4 tiles, [a2, b2) KJ = 2 tiles,
    int32_t a1, b1, a8, b8;     // [a1, b1) KJ = 1 tiles, [a8, b8) KJ = 8 tiles (instances with 129..256 jobs)
};

struct JssParams {
    int32_t n_envs, Jcap, Mcap, block_words;   // Jcap / Mcap / block_words: batch maxima (shared-memory sizing only)
    int32_t jobs_max, machines_max, mask_stride, create_flags;
    int32_t uniform_inst;    // >= 0: every env runs this instance and `order` is the identity
    uint64_t env_id_base;
    const JssInstDesc *inst;
    const uint16_t *ops_pool;
    const int32_t *len_pool;
    const uint16_t *rem_pool;
    const int32_t *order;    // env ids grouped by (KJ class, instance)
    const JssTile *tiles;
    const JssCtaRange *cta_ranges;   // mixed-batch step kernel: per CTA an equal slice of every lane class
    int32_t n_cta_ranges;
    const uint32_t *state_off16;   // per env: start of its state block, in 16-byte units (tile order, see JssTile)
    const uint32_t *hdr_off16;     // per env: start of its 4-word header (t, flags, episode steps / return), 16-byte units
    int32_t *state;          // per-env blocks of 5 * Jcap_i + Mcap_i + 12 words (Jcap_i, Mcap_i: the env's instance)
    uint8_t *mask;           // [N][mask_stride]
    float *obs;              // [N][jobs_max][7]
    int32_t *scalars;        // [N][4]: reward (f32 bits), raw reward, current_time_step, flags << 8 | done
    int32_t *solution;       // [N][jobs_max][machines_max] or nullptr
    int32_t *episode_count;
    int32_t *last_makespan;
    int32_t *last_return;
    int64_t *acc;            // [N][4]: total finished-episode steps, sum makespan, sum return, (min<<32|max) packed
    // canonical export buffers
    int32_t *x_todo, *x_tufco, *x_idle_last, *x_total_idle, *x_col4, *x_tuam;
    uint8_t *x_legal, *x_blocked;
};

// Per-instance scalars: staged in shared memory next to the tables (CTA-uniform, re-read with cheap
// broadcast LDS instead of pinning ~14 registers per thread), or -- uniform batches -- passed in the
// kernel parameters so they become constant-bank operands.
struct SmInst {
    int J, M, max_time_op, max_time_jobs, sum_op;
    float f_mto, f_mtj, f_sop, f_M;       // the divisors as floats ...
    float r_mto, r_mtj, r_sop, r_M;       // ... and their correctly rounded reciprocals
    int Jcap, Mcap, block_words;          // state-block geometry of THIS instance: J, M rounded up to 4; 5*Jcap + Mcap + 12
    // NEGATED divisor / reciprocal PAIRS for the packed (f32x2) observation quotients: columns (1,4), (2,3), (5,6)
    float n14[2], r14[2], n23[2], r23[2], n56[2], r56[2];
    int pad_[4];                          // 32 words: the tables behind it in shared memory stay 16-byte aligned
};
static_assert(sizeof(SmInst) % 16 == 0, "SmInst must keep the shared-memory tables 16-byte aligned");
struct JssLaunch {           // per-launch arguments
    int32_t tile_begin, tile_end;
    int32_t mode;            // JSS_MODE_*
    int32_t rule, coin_mode, n_steps, write_obs;
    int32_t export_after;    // step through the generic kernel: also decode the new state into the x_* arrays (facade)
    uint64_t seed, step_index;
    uint32_t hash_key;       // jss_hash_key(seed, step_index), folded once per launch on the host (fused step + sampler)
    uint32_t pad_key_;
    double cr_factor;        // CriticalRatio due_date_factor (dispatching.py:337-349); reference default 1.5
    const int32_t *actions;  // step
    int32_t *actions_out;    // policy
    const uint8_t *env_mask; // reset / import
    // rollout with trajectory recording: outputs of step k of env e go to slot k * n_envs + e of these buffers
    float *traj_obs; uint8_t *traj_mask; int32_t *traj_scalars; int32_t *traj_actions;
    uint8_t *wire;           // pack: [N][wire_stride] packed observation rows (JSS_WIRE_JOB_BYTES per job)
    int32_t wire_stride;
    SmInst uni;              // scalars of the single instance of a uniform batch (step kernel, UNI = true)
};

// Generator mode (jss_assign_generated): every env has its own instance tables in HBM, regenerated on the device at
// each of its resets.  Per env, `tables + env * tbl_bytes` holds [JssInstDesc, padded to 64 B][ops u16][len i32] (the
// unit the step kernel prefetches with one bulk copy), `rem + env * rem_elems` the suffix sums, `index[env]` the number
// k of the instance it runs (-1 before the first reset).  The kernels of this mode take it as an extra parameter.
#define JSS_GEN_HDR_BYTES 64
struct JssGenParams {
    int32_t J, M, dmin, dmax;
    uint64_t seed;
    char *tables;
    uint16_t *rem;
    int32_t *index;
    int32_t tbl_bytes;      // 64 + ops_bytes + 4 * round_up(J, 4)
    int32_t ops_bytes;      // 2 * round_up(J * M, 8)
    int32_t rem_elems;      // round_up(J * (M + 1), 8)
    int32_t n_envs;
    int32_t warp_stride;    // bytes per warp region: step kernel [step-kernel region][SmInst][tables x 2], generic [SmInst][scratch]
    int32_t off_gen;        // step kernel: offset of [SmInst][tables x 2] inside the warp region
};

#define JSS_MODE_RESET 0
#define JSS_MODE_STEP 1
#define JSS_MODE_ROLLOUT 2
#define JSS_MODE_POLICY 3
#define JSS_MODE_EXPORT 4
#define JSS_MODE_IMPORT 5
#define JSS_MODE_PACK 6     // packed observation wire rows for the host-buffer path (jss_host_step_begin_packed)

#ifndef JSS_WARPS_PER_CTA
#define JSS_WARPS_PER_CTA 8
#endif
