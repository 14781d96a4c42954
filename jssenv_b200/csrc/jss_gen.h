// Random instance generator shared by the device kernels (generator mode, jss_assign_generated) and the host
// restatement jss_generate_instance(), plus the derivation of the packed tables and scalars of one instance that
// jss_load_instances and the device generator both use.  One integer code path for host and device, so instance k of
// global env g under seed s is the same on both (include/jss_b200.h, "generator mode").
//
//   h(c)          = jss_hash3(s ^ JSS_GEN_DOMAIN, g, c)
//   c(j, i, w)    = (k << 20) | (((j * M + i) << 1) | w)
//   duration[j][i] = dmin + jss_pick(h(c(j, i, 0)), dmax - dmin + 1)
//   machine[j]    = Fisher-Yates shuffle of 0..M-1 (Taillard): from the identity, for i = 0 .. M-2
//                   swap positions i and i + jss_pick(h(c(j, i, 1)), M - i)
#pragma once
#include <stdint.h>

#include "jss_rng.h"
#include "jss_types.h"

// keeps instance draws uncorrelated with the policy RNG (jss_hash3(seed, g, step)) when both seeds are equal
#define JSS_GEN_DOMAIN 0x6A09E667F3BCC909ull
#define JSS_GEN_MAX_JOBS 128   // lane classes KJ = 1, 2, 4

JSS_HD static inline uint32_t jss_gen_hash(uint64_t seed, uint64_t genv, uint64_t k, int j, int i, int w, int M) {
    return jss_hash3(seed ^ JSS_GEN_DOMAIN, genv, (k << 20) | (uint64_t)((((j * M + i) << 1) | w)));
}

// row j of instance k: machine order and durations (M <= 32)
JSS_HD static inline void jss_gen_row(uint64_t seed, uint64_t genv, uint64_t k, int j, int M, int dmin, int dmax,
                                      uint8_t *mach, int32_t *dur) {
    const uint32_t span = (uint32_t)(dmax - dmin + 1);
    for (int i = 0; i < M; i++) {
        mach[i] = (uint8_t)i;
        dur[i] = dmin + (int32_t)jss_pick(jss_gen_hash(seed, genv, k, j, i, 0, M), span);
    }
    for (int i = 0; i < M - 1; i++) {
        const int r = i + (int)jss_pick(jss_gen_hash(seed, genv, k, j, i, 1, M), (uint32_t)(M - i));
        const uint8_t t = mach[i];
        mach[i] = mach[r];
        mach[r] = t;
    }
}

// Packed tables of one job row (see jss_types.h): ops[i] = machine << 11 | duration, rem[i] = sum of durations of
// ops i..M-1 (rem[M] = 0).  Returns jobs_length (jss_env.py:87); *max_op receives the row's longest op.
template <typename TM>
JSS_HD static inline int32_t jss_pack_job_row(const TM *mach, const int32_t *dur, int M, uint16_t *ops, uint16_t *rem,
                                              int32_t *max_op) {
    int32_t total = 0, mx = 0;
    for (int i = 0; i < M; i++) {
        ops[i] = (uint16_t)(((uint32_t)mach[i] << JSS_OP_SHIFT) | (uint32_t)dur[i]);
        total += dur[i];
        mx = dur[i] > mx ? dur[i] : mx;
    }
    int32_t suffix = 0;
    rem[M] = 0;
    for (int i = M - 1; i >= 0; i--) {
        suffix += dur[i];
        rem[i] = (uint16_t)suffix;   // <= 32 * 2047 < 65536
    }
    *max_op = mx;
    return total;
}

// descriptor of an instance from its scalars (jss_env.py:86-89); the reciprocals are IEEE divisions on host and
// device alike.  Pool offsets are left 0 for the caller.
JSS_HD static inline JssInstDesc jss_inst_desc(int J, int M, int32_t max_time_op, int32_t max_time_jobs, int32_t sum_op) {
    JssInstDesc d{};
    d.J = J; d.M = M;
    d.max_time_op = max_time_op; d.max_time_jobs = max_time_jobs; d.sum_op = sum_op;
    d.r_mto = 1.0f / (float)max_time_op;
    d.r_mtj = 1.0f / (float)max_time_jobs;
    d.r_sop = 1.0f / (float)sum_op;
    d.r_M = 1.0f / (float)M;
    return d;
}
