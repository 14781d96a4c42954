// jss_device.cuh -- sm_100a device code of the batched job-shop environment.
//
// One warp simulates one environment.  Lane l owns the KJ = 1, 2, 4 (or, for 129..256 jobs, 8) consecutive jobs
// KJ*l .. KJ*l+KJ-1 (so its slice of every per-job array is ONE 4/8/16-byte vector
// load/store and its slice of real_obs is 7 consecutive vectors), and lane m (< M <= 32)
// owns machine m.  A lane keeps the legal / no-op-blocked bits of its own jobs in one
// register (`lb`: bits 0..3 legal, bits 4..7 blocked); warp-wide facts are obtained with
// single VOTE / REDUX instructions.  Everything the reference keeps redundantly (event
// queue, illegal_actions[M][J], machine_legal, counters, needed_machine, total_perform)
// is re-derived in registers (SURVEY.md section 8 a13, appendix A).
//
// Reference semantics implemented here (file:line relative to the reference):
//   env_reset_regs      JSSEnv/envs/jss_env.py:145-181  reset
//   env_advance         JSSEnv/envs/jss_env.py:495-637  increase_time_step
//   env_prioritize      JSSEnv/envs/jss_env.py:183-254  _prioritization_non_final
//   env_check_no_op     JSSEnv/envs/jss_env.py:256-401  _check_no_op
//   env_step            JSSEnv/envs/jss_env.py:403-481  step (+483-493, 639-653)
//   env_emit_*          JSSEnv/envs/jss_env.py:102-134  observation / mask
//   env_select_action   JSSEnv/dispatching.py:92-408    rules; README.md:58-60 sampler
//
// The same source is compiled for the host by tests/emu (32 fibers per warp,
// collectives emulated) so the logic can be differential-tested against the
// oracle without a GPU; that build is test-only and is never loaded by the
// product library.
#pragma once
#include <stdint.h>
#include <string.h>

#include "../../include/jss_b200.h"
#include "jss_gen.h"
#include "jss_rng.h"
#include "jss_types.h"

#define JSS_FULL 0xffffffffu
#define JSS_INF 0x7fffffff

#ifndef JSS_DEV
#define JSS_DEV __device__ __forceinline__
#endif

struct InstView {  // instance tables staged in shared memory
    const uint16_t *ops;
    const int32_t *len;
    const uint16_t *rem;
    const SmInst *si;
    // Shape of the instance for branch conditions and loop bounds.  Uniform-batch kernels point `si` at the kernel
    // parameters (constant bank: ptxas knows those are warp-uniform) and read it there; kernels that stage the instance
    // in shared memory keep register copies that went through jss_uniform (jss_iv_shape).
    int Ju, Mu;
    bool staged;       // compile-time constant after inlining
};
JSS_DEV int jss_J(const InstView &iv) { return iv.staged ? iv.Ju : iv.si->J; }
JSS_DEV int jss_M(const InstView &iv) { return iv.staged ? iv.Mu : iv.si->M; }

template <int KJ>
struct EnvRegs {
    int todo[KJ], tufco[KJ], idle_last[KJ], total_idle[KJ], col4[KJ];
    uint32_t op[KJ];   // packed current op of each owned job, JSS_OP_NONE if none
    uint32_t lb;       // this lane's jobs: bit i = legal, bit 4+i = blocked by a no-op
    int tuam;          // lane m: time_until_available_machine[m]
    int t;             // current_time_step
    uint32_t flags;
    int ep_steps, ep_return;
};

// ---- warp-uniformity hints -----------------------------------------------------------
// ptxas proves a warp converged only while every branch on the way depends on values it KNOWS to be warp-uniform
// (kernel parameters, blockIdx, results of vote / redux / a shuffle from a fixed lane).  One branch on a value it
// cannot classify -- threadIdx.x >> 5, a word every lane loaded from the same shared-memory address -- and every
// *_sync collective after it is compiled as "maybe diverged": UMOV + BRA.DIV + an out-of-line WARPSYNC stub per
// collective, BSSY/BSYNC around each branch, nothing kept in uniform registers.  Passing the few truly uniform
// inputs of an env-step through a lane-0 shuffle removes all of that (mixed-batch step kernel: 75 BRA.DIV sites
// -> 0, 7 344 -> 5 392 SASS instructions, 94 -> 85 us per launch; tests/test_abi_and_host.py pins the property).
// The value MUST be the same in every lane -- the shuffle is a hint, not a broadcast of lane 0's opinion.
JSS_DEV int jss_uniform(int v) {
#ifdef JSS_NO_UNIFORM_HINTS
    return v;
#else
    return __shfl_sync(JSS_FULL, v, 0);
#endif
}
JSS_DEV uint32_t jss_uniform(uint32_t v) { return (uint32_t)jss_uniform((int)v); }
JSS_DEV int jss_warp_index() { return jss_uniform((int)(threadIdx.x >> 5)); }
// Where the flags word gets the hint.  Measured on B200 (profiles/r02_notes.md, session 8): every step / rollout kernel
// gains 9..12 % except the uniform 4-jobs-per-lane step kernel (the ta71..80 shape), which executes 9 % fewer
// instructions with the hint but stalls longer on the TMA command flush and the mbarrier poll and ends up 2 % slower
// (94.5 vs 92.3 us per 65 536-env launch) -- that one instantiation keeps the conservative code.
template <int KJ, bool UNI>
JSS_DEV constexpr bool jss_hint_flags() {
#ifdef JSS_EXP_HINT_ALL
    return true;
#else
    return !(UNI && KJ == 4);
#endif
}

// ---- small helpers --------------------------------------------------------------
template <int KJ, typename T>
JSS_DEV T jss_sel(const T (&a)[KJ], int i) {  // a[i] without dynamic register indexing
    T r = a[0];
#pragma unroll
    for (int k = 1; k < KJ; k++) r = (i == k) ? a[k] : r;
    return r;
}
// (mask >> pos) & 1 for pos that may be >= 32 (JSS_OP_NONE): the hardware shift clamps,
// the host emulation needs the explicit test
JSS_DEV uint32_t jss_bit(uint32_t mask, uint32_t pos) {
#ifdef JSS_EMU
    return pos < 32u ? (mask >> pos) & 1u : 0u;
#else
    return __funnelshift_rc(mask, 0u, pos) & 1u;   // SHF.R with the shift clamped to 32
#endif
}
JSS_DEV uint32_t jss_op_m(uint32_t op) { return op >> JSS_OP_SHIFT; }
JSS_DEV int jss_op_d(uint32_t op) { return (int)(op & JSS_OP_DMASK); }
template <int KJ>
JSS_DEV constexpr uint32_t jss_legal_mask() { return (1u << KJ) - 1u; }
// `lb` layout: bit i = job slot i legal, bit BS + i = blocked by a no-op (BS = 4 for KJ <= 4, 8 for KJ = 8); a lane's
// bits are one byte of the state block (KJ <= 4) or one 16-bit word (KJ = 8: 129..256 jobs)
template <int KJ>
JSS_DEV constexpr int jss_bs() { return KJ == 8 ? 8 : 4; }
template <int KJ>
JSS_DEV constexpr int jss_bits_words() { return KJ == 8 ? 16 : 8; }   // int32 words of the per-lane bits region

// correctly rounded x / y for small non-negative integers given ry = RN(1/y): Markstein's
// sequence q = RN(x*ry); r = x - q*y (exact, FMA); q' = RN(q + r*ry).  Checked exhaustively
// against IEEE division for every (x, y) the bundled instances can produce and all y <= 4096
// (tools/check_div.c); replaces the ~25-instruction IEEE fp32 division and its slow path.
JSS_DEV float jss_div(float x, float y, float ry) {
    const float q = __fmul_rn(x, ry);
    const float r = __fmaf_rn(-q, y, x);
    return __fmaf_rn(r, ry, q);
}

// two quotients at once on the packed-fp32 pipe (sm_100 FMUL2 / FFMA2): the same three roundings per element
// as jss_div, so the results are identical
#ifndef JSS_EMU
JSS_DEV float2 jss_div2(float2 x, const float (&ny)[2], const float (&ry)[2]) {   // ny = -divisor (host-negated)
    unsigned long long xx, nn, rr, q, e, o;
    xx = *reinterpret_cast<unsigned long long *>(&x);
    const float2 nv = make_float2(ny[0], ny[1]), rv = make_float2(ry[0], ry[1]);
    nn = *reinterpret_cast<const unsigned long long *>(&nv);
    rr = *reinterpret_cast<const unsigned long long *>(&rv);
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(q) : "l"(xx), "l"(rr));
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(e) : "l"(q), "l"(nn), "l"(xx));      // x - q * y, exact
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(o) : "l"(e), "l"(rr), "l"(q));
    return *reinterpret_cast<float2 *>(&o);
}
#else
JSS_DEV float2 jss_div2(float2 x, const float (&ny)[2], const float (&ry)[2]) {
    return make_float2(jss_div(x.x, -ny[0], ry[0]), jss_div(x.y, -ny[1], ry[1]));
}
#endif

// ---- TMA (cp.async.bulk) + mbarrier helpers -----------------------------------------------
// The state block of the NEXT env of a warp is prefetched into the warp's shared-memory
// buffer by one bulk copy (global -> shared, completion on an mbarrier) while the current env
// is simulated; an env's observation rows leave shared memory with one bulk copy
// (shared -> global).  Sizes/addresses are multiples of 16 bytes by construction.
// Shared-memory operands are passed as 32-bit shared-space addresses (jss_saddr_t) computed from
// ONE base register, so no generic<->shared address conversions are needed at the call sites.
#ifndef JSS_EMU
typedef uint32_t jss_saddr_t;
JSS_DEV jss_saddr_t jss_saddr(const void *generic_ptr) { return (uint32_t)__cvta_generic_to_shared(generic_ptr); }
JSS_DEV void jss_mbar_init(jss_saddr_t mbar) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(mbar) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
JSS_DEV void jss_bulk_load(jss_saddr_t smem_dst, const void *gmem_src, uint32_t bytes, jss_saddr_t mbar) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_dst), "l"(gmem_src), "r"(bytes), "r"(mbar) : "memory");
}
JSS_DEV void jss_mbar_wait(jss_saddr_t mbar, uint32_t phase) {
    uint32_t ok;
    do {
        // non-blocking poll: test_wait returns at once, try_wait may park the warp for a scheduler time slice when the
        // block has not landed yet (measured: test_wait 0.3-0.7 % faster on the uniform and mixed step kernels)
#ifdef JSS_MBAR_TRY_WAIT
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                     : "=r"(ok) : "r"(mbar), "r"(phase) : "memory");
#else
        asm volatile("{\n .reg .pred p;\n mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                     : "=r"(ok) : "r"(mbar), "r"(phase) : "memory");
#endif
    } while (!ok);
}
JSS_DEV void jss_fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
JSS_DEV void jss_fence_async_global() { asm volatile("fence.proxy.async.global;" ::: "memory"); }
JSS_DEV void jss_bulk_store(void *gmem_dst, jss_saddr_t smem_src, uint32_t bytes) {   // joins the open bulk group
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                 ::"l"(gmem_dst), "r"(smem_src), "r"(bytes) : "memory");
#ifdef JSS_EXP_TWO_COMMITS
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
#endif
}
JSS_DEV void jss_bulk_commit() {
#ifndef JSS_EXP_TWO_COMMITS
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
#endif
}
JSS_DEV void jss_bulk_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
JSS_DEV void jss_bulk_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// several bulk loads completing on ONE mbarrier phase: one arrive announcing the total, then the copies
JSS_DEV void jss_mbar_expect_tx(jss_saddr_t mbar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
}
JSS_DEV void jss_bulk_copy(jss_saddr_t smem_dst, const void *gmem_src, uint32_t bytes, jss_saddr_t mbar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_dst), "l"(gmem_src), "r"(bytes), "r"(mbar) : "memory");
}
#else   // host emulation (tests/emu): synchronous copies; the waits are warp rendezvous points
typedef char *jss_saddr_t;
JSS_DEV jss_saddr_t jss_saddr(const void *generic_ptr) { return (char *)generic_ptr; }
JSS_DEV void jss_mbar_init(jss_saddr_t) {}
JSS_DEV void jss_bulk_load(jss_saddr_t smem_dst, const void *gmem_src, uint32_t bytes, jss_saddr_t) { memcpy(smem_dst, gmem_src, bytes); }
JSS_DEV void jss_mbar_wait(jss_saddr_t, uint32_t) { __syncwarp(); }
JSS_DEV void jss_fence_async_smem() {}
JSS_DEV void jss_fence_async_global() {}
JSS_DEV void jss_bulk_store(void *gmem_dst, jss_saddr_t smem_src, uint32_t bytes) { memcpy(gmem_dst, smem_src, bytes); }
JSS_DEV void jss_bulk_commit() {}
JSS_DEV void jss_bulk_store_wait_read() {}
JSS_DEV void jss_bulk_store_wait_all() {}
JSS_DEV void jss_mbar_expect_tx(jss_saddr_t, uint32_t) {}
JSS_DEV void jss_bulk_copy(jss_saddr_t smem_dst, const void *gmem_src, uint32_t bytes, jss_saddr_t) { memcpy(smem_dst, gmem_src, bytes); }
#endif

// vector access to a lane's KJ-word slice
template <int KJ>
JSS_DEV void jss_ld(const int32_t *p, int (&o)[KJ]);
template <>
JSS_DEV void jss_ld<1>(const int32_t *p, int (&o)[1]) { o[0] = *p; }
template <>
JSS_DEV void jss_ld<2>(const int32_t *p, int (&o)[2]) {
    int2 v = *reinterpret_cast<const int2 *>(p);
    o[0] = v.x; o[1] = v.y;
}
template <>
JSS_DEV void jss_ld<4>(const int32_t *p, int (&o)[4]) {
    int4 v = *reinterpret_cast<const int4 *>(p);
    o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w;
}
template <>
JSS_DEV void jss_ld<8>(const int32_t *p, int (&o)[8]) {
    const int4 a = reinterpret_cast<const int4 *>(p)[0], b = reinterpret_cast<const int4 *>(p)[1];
    o[0] = a.x; o[1] = a.y; o[2] = a.z; o[3] = a.w; o[4] = b.x; o[5] = b.y; o[6] = b.z; o[7] = b.w;
}
template <int KJ>
JSS_DEV void jss_st(int32_t *p, const int (&o)[KJ]);
template <>
JSS_DEV void jss_st<1>(int32_t *p, const int (&o)[1]) { *p = o[0]; }
template <>
JSS_DEV void jss_st<2>(int32_t *p, const int (&o)[2]) { *reinterpret_cast<int2 *>(p) = make_int2(o[0], o[1]); }
template <>
JSS_DEV void jss_st<4>(int32_t *p, const int (&o)[4]) {
    *reinterpret_cast<int4 *>(p) = make_int4(o[0], o[1], o[2], o[3]);
}

template <>
JSS_DEV void jss_st<8>(int32_t *p, const int (&o)[8]) {
    reinterpret_cast<int4 *>(p)[0] = make_int4(o[0], o[1], o[2], o[3]);
    reinterpret_cast<int4 *>(p)[1] = make_int4(o[4], o[5], o[6], o[7]);
}

// a lane's legal / blocked bits inside the state block
template <int KJ>
JSS_DEV uint32_t jss_ld_bits(const int32_t *bits_region, int lane) {
    if (KJ == 8) return reinterpret_cast<const uint16_t *>(bits_region)[lane];
    return reinterpret_cast<const uint8_t *>(bits_region)[lane];
}
template <int KJ>
JSS_DEV void jss_st_bits(int32_t *bits_region, int lane, uint32_t lb) {
    if (KJ == 8) reinterpret_cast<uint16_t *>(bits_region)[lane] = (uint16_t)lb;
    else reinterpret_cast<uint8_t *>(bits_region)[lane] = (uint8_t)lb;
}

// ---- state block <-> registers -----------------------------------------------------
// Padding slots (job index >= J inside the last active lane, and whole lanes past the
// last job) hold todo == M, i.e. they behave like finished jobs everywhere.
template <int KJ>
JSS_DEV void env_derive_ops(const InstView &iv, EnvRegs<KJ> &s, int lane) {
    const int M = jss_M(iv);
    // lanes past the last job read row 0 (any in-bounds row: their todo == M selects JSS_OP_NONE anyway)
    const int row = (KJ * lane < jss_J(iv)) ? KJ * lane * M : 0;
#pragma unroll
    for (int i = 0; i < KJ; i++) {
        // unconditional load of a clamped index + select: no divergent branch around the table lookup
        const uint32_t o = iv.ops[row + i * M + min(s.todo[i], M - 1)];
        s.op[i] = (s.todo[i] < M) ? o : JSS_OP_NONE;
    }
}

template <int KJ>
JSS_DEV void env_clear_jobs(const InstView &iv, EnvRegs<KJ> &s) {
#pragma unroll
    for (int i = 0; i < KJ; i++) { s.todo[i] = jss_M(iv); s.tufco[i] = 0; s.idle_last[i] = 0; s.total_idle[i] = 0; s.col4[i] = 0; }
}

template <int KJ>
JSS_DEV void env_load_from(const JssParams &p, const InstView &iv, const int32_t *blk, int lane, EnvRegs<KJ> &s) {
    const int Jc = iv.si->Jcap, Mc = iv.si->Mcap;   // geometry of the env's own instance
    if (KJ * lane < jss_J(iv)) {
        const int32_t *q = blk + KJ * lane;
        jss_ld<KJ>(q, s.todo);
        jss_ld<KJ>(q + Jc, s.tufco);
        jss_ld<KJ>(q + 2 * Jc, s.idle_last);
        jss_ld<KJ>(q + 3 * Jc, s.total_idle);
        jss_ld<KJ>(q + 4 * Jc, s.col4);
    } else {
        env_clear_jobs<KJ>(iv, s);
    }
    const int32_t *tail = blk + 5 * Jc;
    s.tuam = (lane < jss_M(iv)) ? tail[lane] : 0;
    s.lb = jss_ld_bits<KJ>(tail + Mc, lane);
    const int4 h4 = *reinterpret_cast<const int4 *>(tail + Mc + jss_bits_words<KJ>());
    s.t = h4.x; s.flags = (uint32_t)h4.y; s.ep_steps = h4.z; s.ep_return = h4.w;
    env_derive_ops<KJ>(iv, s, lane);
}
// start of env's state block (blocks are stored in tile order with per-instance sizes, see JssTile)
JSS_DEV int32_t *env_block(const JssParams &p, int env) { return p.state + (size_t)p.state_off16[env] * 4; }
template <int KJ>
JSS_DEV void env_load(const JssParams &p, const InstView &iv, int env, int lane, EnvRegs<KJ> &s) {
    env_load_from<KJ>(p, iv, env_block(p, env), lane, s);
}

// policy kernels read only what the rule looks at: bits + header always, todo for every
// rule (current op / remaining work / remaining ops), idle_last for FIFO
template <int KJ>
JSS_DEV void env_load_for_policy(const JssParams &p, const InstView &iv, int env, int lane, EnvRegs<KJ> &s,
                                 int rule) {
    const int32_t *blk = env_block(p, env);
    const int Jc = iv.si->Jcap, Mc = iv.si->Mcap;
    env_clear_jobs<KJ>(iv, s);
    if (rule != JSS_RULE_RANDOM && KJ * lane < jss_J(iv)) {
        jss_ld<KJ>(blk + KJ * lane, s.todo);
        if (rule == JSS_RULE_FIFO) jss_ld<KJ>(blk + 2 * Jc + KJ * lane, s.idle_last);
    }
    s.tuam = 0;
    const int32_t *tail = blk + 5 * Jc;
    s.lb = jss_ld_bits<KJ>(tail + Mc, lane);
    const int4 h4 = *reinterpret_cast<const int4 *>(tail + Mc + jss_bits_words<KJ>());
    s.t = h4.x; s.flags = (uint32_t)h4.y; s.ep_steps = h4.z; s.ep_return = h4.w;
    if (rule != JSS_RULE_RANDOM) env_derive_ops<KJ>(iv, s, lane);
    else {
#pragma unroll
        for (int i = 0; i < KJ; i++) s.op[i] = JSS_OP_NONE;
    }
}

template <int KJ>
JSS_DEV void env_store_to(const JssParams &p, const InstView &iv, int32_t *blk, int lane, const EnvRegs<KJ> &s) {
    const int Jc = iv.si->Jcap, Mc = iv.si->Mcap;
    if (KJ * lane < Jc) {       // lanes past the last job hold the "finished job" padding values: the whole block is defined
        int32_t *q = blk + KJ * lane;
        jss_st<KJ>(q, s.todo);
        jss_st<KJ>(q + Jc, s.tufco);
        jss_st<KJ>(q + 2 * Jc, s.idle_last);
        jss_st<KJ>(q + 3 * Jc, s.total_idle);
        jss_st<KJ>(q + 4 * Jc, s.col4);
    }
    int32_t *tail = blk + 5 * Jc;
    if (lane < Mc) tail[lane] = (lane < jss_M(iv)) ? s.tuam : 0;
    jss_st_bits<KJ>(tail + Mc, lane, s.lb);
    if (lane == 0)
        *reinterpret_cast<int4 *>(tail + Mc + jss_bits_words<KJ>()) = make_int4(s.t, (int)s.flags, s.ep_steps, s.ep_return);
}

template <int KJ>
JSS_DEV void env_store(const JssParams &p, const InstView &iv, int env, int lane, const EnvRegs<KJ> &s) {
    // all lanes must have finished env_load (every lane reads the shared header words)
    // before any lane overwrites the block: paths such as the auto-reset have no
    // collective between load and store
    __syncwarp();
    env_store_to<KJ>(p, iv, env_block(p, env), lane, s);
}

// jss_env.py:145-181
template <int KJ>
JSS_DEV void env_reset_regs(const InstView &iv, EnvRegs<KJ> &s, int lane) {
    s.lb = 0u;
#pragma unroll
    for (int i = 0; i < KJ; i++) {
        const bool valid = KJ * lane + i < jss_J(iv);
        s.todo[i] = valid ? 0 : jss_M(iv);
        s.tufco[i] = 0; s.idle_last[i] = 0; s.total_idle[i] = 0; s.col4[i] = 0;
        if (valid) s.lb |= 1u << i;               // every job legal, no-op illegal (:160-161)
    }
    s.tuam = 0; s.t = 0; s.flags = 0u; s.ep_steps = 0; s.ep_return = 0;
    env_derive_ops<KJ>(iv, s, lane);
}

// ---- increase_time_step (jss_env.py:495-637); returns hole_planning ---------------
template <int KJ>
JSS_DEV int env_advance(const InstView &iv, EnvRegs<KJ> &s, int lane) {
    // next event = smallest positive machine countdown (the sorted event list of
    // the reference always equals {t + tuam[m] : tuam[m] > 0}, appendix A.1)
    const int tuam_old = s.tuam;
    const int diff = (int)__reduce_min_sync(JSS_FULL, (unsigned)(tuam_old > 0 ? tuam_old : JSS_INF));
    const int gap = diff - tuam_old;                      // > 0 only for machines idle before the event
    const int hole = (int)__reduce_add_sync(JSS_FULL, (unsigned)((lane < jss_M(iv) && gap > 0) ? gap : 0));
    s.t += diff;
    const int M = jss_M(iv);
    const int row = (KJ * lane < jss_J(iv)) ? KJ * lane * M : 0;   // lanes past the last job: any in-bounds row
#pragma unroll
    for (int i = 0; i < KJ; i++) {
        // branch-free form of the reference's three cases (select instructions instead of divergent
        // branches): running (:529), running and finishing now (:550), waiting (:594); finished jobs
        // (todo == M) fall through unchanged
        const int was = s.tufco[i];
        const int left = was - diff;
        const bool running = was > 0;
        const bool finished = running && left <= 0;
        const bool waiting = !running && s.todo[i] < M;
        s.tufco[i] = left > 0 ? left : 0;                 // == max(0, was - diff); 0 stays 0
        const int slack = diff - was;                     // idle part of the step for a job finishing now
        s.total_idle[i] += finished ? slack : (waiting ? diff : 0);
        s.idle_last[i] = finished ? slack : s.idle_last[i] + (waiting ? diff : 0);
        s.todo[i] += finished ? 1 : 0;
        {   // next op of a job that just finished one: unconditional clamped lookup + selects (no branch)
            const uint32_t o = iv.ops[row + i * M + min(s.todo[i], M - 1)];
            s.op[i] = finished ? ((s.todo[i] < M) ? o : JSS_OP_NONE) : s.op[i];
        }
        // real_obs[:,4] uses the PRE-decrement countdown of the next machine (:569-578)
        const int tq = __shfl_sync(JSS_FULL, tuam_old, (int)(jss_op_m(s.op[i]) & 31u));
        const int w = tq - diff;
        const int c4 = (s.op[i] != JSS_OP_NONE) ? (w > 0 ? w : 0) : iv.si->max_time_op;   // max_time_op encodes 1.0 (:586)
        s.col4[i] = finished ? c4 : s.col4[i];
    }
    s.tuam = gap < 0 ? -gap : 0;
    const uint32_t free_m = __ballot_sync(JSS_FULL, lane < jss_M(iv) && s.tuam == 0);
#pragma unroll
    for (int i = 0; i < KJ; i++)                          // legalisation (:616-634): free machine and not blocked
        s.lb |= (jss_bit(free_m, jss_op_m(s.op[i])) & ~(s.lb >> (jss_bs<KJ>() + i)) & 1u) << i;
    return hole;
}

// machines that have at least one legal job (== machine_legal of the reference)
template <int KJ>
JSS_DEV uint32_t env_machine_legal(const EnvRegs<KJ> &s) {
    uint32_t mine = 0u;
#pragma unroll
    for (int i = 0; i < KJ; i++) mine |= ((s.lb >> i) & 1u) << (jss_op_m(s.op[i]) & 31u);
    return __reduce_or_sync(JSS_FULL, mine);
}

// ---- _prioritization_non_final (jss_env.py:183-254) --------------------------------
template <int KJ>
JSS_DEV void env_prioritize(const InstView &iv, EnvRegs<KJ> &s, int lane) {
    uint32_t fin = 0u;                                    // my legal FINAL ops
    const int last = jss_M(iv) - 1;
#pragma unroll
    for (int i = 0; i < KJ; i++) fin |= (s.todo[i] == last ? 1u : 0u) << i;
    fin &= s.lb;
    if (!__any_sync(JSS_FULL, fin != 0u)) return;         // nothing can be de-legalised (the common case)
    uint32_t fin_m = 0u;                                  // machines wanted by a legal final op
#pragma unroll
    for (int i = 0; i < KJ; i++)
        if (fin & (1u << i)) fin_m |= 1u << (jss_op_m(s.op[i]) & 31u);
    fin_m = __reduce_or_sync(JSS_FULL, fin_m);
    const uint32_t free_m = __ballot_sync(JSS_FULL, lane < jss_M(iv) && s.tuam == 0);
    int cand_d[KJ];                                       // duration if legal non-final op whose NEXT machine is free
    const int row = KJ * lane * jss_M(iv);
#pragma unroll
    for (int i = 0; i < KJ; i++) {
        cand_d[i] = JSS_INF;
        if ((s.lb & (1u << i)) && !(fin & (1u << i))) {
            const uint32_t nxt = iv.ops[row + i * jss_M(iv) + s.todo[i] + 1];
            if (jss_bit(free_m, jss_op_m(nxt))) cand_d[i] = jss_op_d(s.op[i]);   // :234-239
        }
    }
    uint32_t kill = 0u;
    while (fin_m) {                                       // per machine with a legal final op
        const uint32_t m = (uint32_t)(__ffs((int)fin_m) - 1);
        fin_m &= fin_m - 1u;
        int mn = JSS_INF;
#pragma unroll
        for (int i = 0; i < KJ; i++)
            if (cand_d[i] != JSS_INF && jss_op_m(s.op[i]) == m) mn = min(mn, cand_d[i]);
        mn = (int)__reduce_min_sync(JSS_FULL, (unsigned)mn);   // min_non_final (:238)
        if (mn != JSS_INF) {
#pragma unroll
            for (int i = 0; i < KJ; i++)
                if ((fin & (1u << i)) && jss_op_m(s.op[i]) == m && jss_op_d(s.op[i]) > mn) kill |= 1u << i;  // :252
        }
    }
    s.lb &= ~kill;
}

// ---- _check_no_op (jss_env.py:256-401); returns legal_actions[J] -----------------
// `hz` is a 32-int per-warp shared scratch (aliases the observation staging area).
template <int KJ>
JSS_DEV bool env_check_no_op(const InstView &iv, const EnvRegs<KJ> &s, int lane, uint32_t ML, int nlegal,
                             int *hz) {
    const unsigned mn = __reduce_min_sync(JSS_FULL, (unsigned)(s.tuam > 0 ? s.tuam : JSS_INF));
    if (mn == (unsigned)JSS_INF || __popc(ML) > 3 || nlegal > 4) return false;   // gate :284-288
    const int next_event = s.t + (int)mn;                                        // :293
    int maxh = s.t;                                                              // :296
    int lm0 = -1, lm1 = -1, lm2 = -1;                   // the <= 3 legal machines and their horizons
    const int hinit = s.t + iv.si->max_time_op;             // :300-302
    int h0 = hinit, h1 = hinit, h2 = hinit;
    // pass 1 (:305-321): legal jobs in ascending job index = ascending lane, then slot
    uint32_t lanes = __ballot_sync(JSS_FULL, (s.lb & jss_legal_mask<KJ>()) != 0u);
    while (lanes) {
        const int l = __ffs((int)lanes) - 1;
        lanes &= lanes - 1u;
        // KJ = 1: the lane's only job is the legal one (no need to fetch its bits, no inner loop)
        uint32_t bits = (KJ == 1) ? 1u : (__shfl_sync(JSS_FULL, s.lb, l) & jss_legal_mask<KJ>());
#pragma unroll 1
        while (bits) {                                  // warp-uniform: the legal jobs of lane l, ascending
            const int i = (KJ == 1) ? 0 : __ffs((int)bits) - 1;
            bits = (KJ == 1) ? 0u : (bits & (bits - 1u));
            const uint32_t o = __shfl_sync(JSS_FULL, jss_sel<KJ>(s.op, i), l);
            const int m = (int)jss_op_m(o);
            const int end = s.t + jss_op_d(o);
            if (end < next_event) return false;         // :314-315
            int cur;
            if (lm0 == m || lm0 < 0) { lm0 = m; h0 = min(h0, end); cur = h0; }
            else if (lm1 == m || lm1 < 0) { lm1 = m; h1 = min(h1, end); cur = h1; }
            else { lm2 = m; h2 = min(h2, end); cur = h2; }
            maxh = max(maxh, cur);                      // :321
        }
    }
    const int last = jss_M(iv) - 1;
    // per-machine horizon table: finite only for machines that have a legal job, so the
    // walk's test `max_horizon_machine[m] > time and machine_legal[m]` is one compare
    hz[lane] = (lane == lm0) ? h0 : (lane == lm1) ? h1 : (lane == lm2) ? h2 : (int)0x80000000;
    __syncwarp();
    // pass 2 (:324-401): jobs that are not legal now but may need a legal machine soon
    uint32_t want = 0u;
    const int row = KJ * lane * jss_M(iv);
#pragma unroll
    for (int i = 0; i < KJ; i++) {
        // countdown of the job's current machine (case 2, :374-377)
        const int tq = __shfl_sync(JSS_FULL, s.tuam, (int)(jss_op_m(s.op[i]) & 31u));
        if (!(s.lb & (1u << i)) && s.todo[i] < jss_M(iv)) {
            int ts, tm;
            if (s.tufco[i] > 0) { ts = s.todo[i] + 1; tm = s.t + s.tufco[i]; }      // case 1 (:327-337); a running
            else if (!(s.lb & ((1u << jss_bs<KJ>()) << i))) { ts = s.todo[i]; tm = s.t + tq; }       // last op walks nothing either way
            else { ts = jss_M(iv); tm = 0; }                                         // case 2 (:366-377) / blocked
            const uint16_t *o_ptr = iv.ops + row + i * jss_M(iv);
            while (ts < last && maxh > tm) {                                        // :340-342 / :380-382
                const uint32_t o = o_ptr[ts];
                if (hz[jss_op_m(o)] > tm) want |= 1u << jss_op_m(o);                // machine_next.add (:351 / :391)
                tm += jss_op_d(o);
                ts += 1;
            }
        }
        // the reference returns as soon as machine_next covers every legal machine (:357 / :395);
        // about half of the pass-2 runs end "legal", most of them after the first job slot
        if (i + 1 < KJ && ML != 0u && __reduce_or_sync(JSS_FULL, want) == ML) {
            __syncwarp();                               // hz aliases the obs staging buffer
            return true;
        }
    }
    want = __reduce_or_sync(JSS_FULL, want);
    __syncwarp();                                       // hz aliases the obs staging buffer
    return ML != 0u && want == ML;                      // len(machine_next) == nb_machine_legal
}

// Output bases of the emit helpers: the library's per-env buffers by default, the caller's trajectory buffers when a
// rollout records (then `env` is the trajectory slot k * N + env).
struct JssOut {
    float *obs;
    uint8_t *mask;
    int32_t *scalars;
};
JSS_DEV JssOut jss_out_default(const JssParams &p) { return JssOut{p.obs, p.mask, p.scalars}; }

// ---- observation / mask / reward (jss_env.py:102-134, 483-493) ---------------------
template <int KJ, bool BULK = false>
JSS_DEV void env_emit_obs(const JssParams &p, const JssOut &out, const InstView &iv, const EnvRegs<KJ> &s, int env, int lane,
                          float *scratch, jss_saddr_t scratch_sa = jss_saddr_t(), void *st_dst = nullptr,
                          jss_saddr_t st_sa = jss_saddr_t(), uint32_t st_bytes = 0u) {
    if (KJ * lane < jss_J(iv)) {
        float v[KJ * 7];
#pragma unroll
        for (int i = 0; i < KJ; i++) {
            // total_perform_op_time_jobs == t - total_idle while the job is unfinished,
            // jobs_length[j] afterwards (every advance adds `difference` to exactly one of
            // the two counters until the job completes)
            const int len = iv.len[KJ * lane + i];        // unconditional (in-bounds) load + select
            const int perf = (s.todo[i] < jss_M(iv)) ? s.t - s.total_idle[i] : len;
            v[7 * i + 0] = (s.lb & (1u << i)) ? 1.0f : 0.0f;
            // columns that share a divisor (or sit next to each other) go through the packed-fp32 pipe in pairs
            const float2 q14 = jss_div2(make_float2((float)s.tufco[i], (float)s.col4[i]), iv.si->n14, iv.si->r14);
            const float2 q23 = jss_div2(make_float2((float)s.todo[i], (float)perf), iv.si->n23, iv.si->r23);
            const float2 q56 = jss_div2(make_float2((float)s.idle_last[i], (float)s.total_idle[i]), iv.si->n56, iv.si->r56);
            v[7 * i + 1] = q14.x; v[7 * i + 4] = q14.y;
            v[7 * i + 2] = q23.x; v[7 * i + 3] = q23.y;
            v[7 * i + 5] = q56.x; v[7 * i + 6] = q56.y;
        }
        // stage the lane's 7*KJ floats (one contiguous, bank-conflict-free run per lane) ...
        float *mine = scratch + 7 * KJ * lane;
        if (KJ == 4 || KJ == 8) {
#pragma unroll
            for (int q = 0; q < 7 * KJ / 4; q++)
                reinterpret_cast<float4 *>(mine)[q] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
        } else if (KJ == 2) {
#pragma unroll
            for (int q = 0; q < 7; q++) reinterpret_cast<float2 *>(mine)[q] = make_float2(v[2 * q], v[2 * q + 1]);
        } else {
#pragma unroll
            for (int q = 0; q < 7; q++) mine[q] = v[q];
        }
    }
    float *dst = out.obs + (size_t)env * p.jobs_max * 7;
    const int n = jss_J(iv) * 7;
    if (BULK) {
        // ONE proxy fence covers both staged buffers (new state block + observation rows), then lane 0
        // hands them to the TMA engine: one bulk copy shared -> global each
        jss_fence_async_smem();          // make the generic-proxy writes visible to the async proxy
        __syncwarp();
        if (lane == 0) {
            if (st_bytes) jss_bulk_store(st_dst, st_sa, st_bytes);
            if ((n & 3) == 0 && (p.jobs_max & 3) == 0) jss_bulk_store(dst, scratch_sa, (uint32_t)n * 4u);
            jss_bulk_commit();           // ONE group for both copies (an empty group is legal)
        }
        if ((n & 3) == 0 && (p.jobs_max & 3) == 0)
            return;                      // the caller waits (wait_group.read) before reusing the staging buffers
    } else {
        __syncwarp();
    }
    // ... and stream the J*7 floats of the env out with fully coalesced stores
    int done_elems = 0;
    if ((p.jobs_max & 3) == 0) {
        const int n4 = n >> 2;
        for (int k = lane; k < n4; k += 32)
            reinterpret_cast<float4 *>(dst)[k] = reinterpret_cast<const float4 *>(scratch)[k];
        done_elems = n4 << 2;
    }
    for (int k = done_elems + lane; k < n; k += 32) dst[k] = scratch[k];
    __syncwarp();
}

template <int KJ>
JSS_DEV void env_emit_mask(const JssParams &p, const JssOut &out, const InstView &iv, const EnvRegs<KJ> &s, int env, int lane,
                           bool noop) {
    uint8_t *row = out.mask + (size_t)env * p.mask_stride;
    const int j0 = KJ * lane;
    if (KJ == 8) {
        if (j0 <= jss_J(iv)) {                            // 8 mask bytes per lane: two 4-bit spreads (rows are 8-byte aligned)
            uint32_t lo = ((s.lb & 15u) * 0x00204081u) & 0x01010101u, hi = (((s.lb >> 4) & 15u) * 0x00204081u) & 0x01010101u;
            const int d = jss_J(iv) - j0;                 // byte J is the no-op flag
            if (d < 4) lo |= (noop ? 1u : 0u) << (8 * d);
            else if (d < 8) hi |= (noop ? 1u : 0u) << (8 * (d - 4));
            *reinterpret_cast<uint2 *>(row + j0) = make_uint2(lo, hi);
        }
    } else if (j0 <= jss_J(iv)) {
        // spread the legal bits to bytes: bit i -> byte i
        // bit i -> byte i: the products of the set bits land on distinct positions (no carries)
        uint32_t w = ((s.lb & jss_legal_mask<KJ>()) * 0x00204081u) & 0x01010101u;
        if (jss_J(iv) - j0 < KJ) w |= (noop ? 1u : 0u) << (8 * (jss_J(iv) - j0));     // byte J is the no-op flag
        if (KJ == 4) *reinterpret_cast<uint32_t *>(row + j0) = w;
        else if (KJ == 2) *reinterpret_cast<uint16_t *>(row + j0) = (uint16_t)w;
        else row[j0] = (uint8_t)w;
    }
    if (jss_J(iv) == 32 * KJ && lane == 0) row[jss_J(iv)] = noop ? 1 : 0;   // no lane owns byte J
}

// reward / raw reward / time / (flags << 8 | done) of an env are ONE 16-byte record, so the
// per-step scalar outputs cost a single store (the API exposes them as strided arrays)
template <int KJ>
JSS_DEV void env_emit_scalars(const JssOut &out, const InstView &iv, const EnvRegs<KJ> &s, int env, int lane,
                              int raw_reward) {
    if (lane == 0) {
        const float r = jss_div((float)raw_reward, iv.si->f_mto, iv.si->r_mto);   // :483-493
        reinterpret_cast<int4 *>(out.scalars)[env] =
            make_int4(__float_as_int(r), raw_reward, s.t, (int)((s.flags << 8) | (s.flags & JSS_FLAG_DONE)));
    }
}

// episode bookkeeping when _is_done() turns true (jss_env.py:649-652)
template <int KJ>
JSS_DEV void env_episode_end(const JssParams &p, const EnvRegs<KJ> &s, int env, int lane) {
    if (lane == 0) {
        const int prev = p.episode_count[env];
        p.episode_count[env] = prev + 1;
        p.last_makespan[env] = s.t;
        p.last_return[env] = s.ep_return;
        int64_t *acc = p.acc + (size_t)env * 4;
        acc[0] += s.ep_steps;
        acc[1] += s.t;
        acc[2] += s.ep_return;
        const uint64_t mm = (uint64_t)acc[3];
        uint32_t mn = prev ? (uint32_t)(mm >> 32) : 0xffffffffu, mx = prev ? (uint32_t)mm : 0u;
        if ((uint32_t)s.t < mn) mn = (uint32_t)s.t;
        if ((uint32_t)s.t > mx) mx = (uint32_t)s.t;
        acc[3] = (int64_t)(((uint64_t)mn << 32) | mx);
    }
}

// ---- step (jss_env.py:403-481) ---------------------------------------------------------
// Returns true if the env changed (outputs must be re-emitted).
template <int KJ>
JSS_DEV bool env_step(const JssParams &p, const InstView &iv, EnvRegs<KJ> &s, int env, int lane, int action,
                      int &raw_reward, int *hz) {
    raw_reward = 0;
    if (action == JSS_ACTION_SKIP) return false;
    if (s.flags & JSS_FLAG_DONE) {
        if (p.create_flags & JSS_CREATE_AUTO_RESET) {
            env_reset_regs<KJ>(iv, s, lane);
            if (p.solution) {
                int32_t *sol = p.solution + (size_t)env * p.jobs_max * p.machines_max;
                for (int k = lane; k < p.jobs_max * p.machines_max; k += 32) sol[k] = -1;
            }
            return true;
        }
        return false;  // frozen until reset
    }
    constexpr uint32_t LM = jss_legal_mask<KJ>();
    int holes = 0, gain = 0;
    const bool wait = (action == JSS_ACTION_ADVANCE || action == jss_J(iv));
    if (wait) {
        if (!__any_sync(JSS_FULL, s.tuam > 0)) { s.flags |= JSS_FLAG_ERROR; return false; }   // IndexError at :517
        if (action == jss_J(iv))                          // no-op (:419-428): legal -> blocked
            s.lb = ((s.lb & LM) << jss_bs<KJ>()) | (s.lb & (LM << jss_bs<KJ>()));
    } else {                                             // job allocation (:441-481)
        if (action < 0 || action > jss_J(iv)) { s.flags |= JSS_FLAG_ERROR; return false; }
        const int la = action / KJ, ia = action % KJ;
        const uint32_t opa = __shfl_sync(JSS_FULL, jss_sel<KJ>(s.op, ia), la);
        const uint32_t bits_a = __shfl_sync(JSS_FULL, s.lb, la);
        if (opa == JSS_OP_NONE || !((bits_a >> ia) & 1u)) { s.flags |= JSS_FLAG_ERROR; return false; }
        const uint32_t m_a = jss_op_m(opa);
        gain = jss_op_d(opa);
        s.tuam = ((uint32_t)lane == m_a) ? gain : s.tuam;            // :446
#pragma unroll
        for (int i = 0; i < KJ; i++) s.tufco[i] = (lane == la && i == ia) ? gain : s.tufco[i];   // :447
        if (p.solution && lane == la)                                 // :454
            p.solution[((size_t)env * p.jobs_max + action) * p.machines_max + jss_sel<KJ>(s.todo, ia)] = s.t;
#pragma unroll
        for (int i = 0; i < KJ; i++)
            // every job waiting for machine m_a: no longer legal (:455-461), no longer
            // no-op-blocked (:464-467; illegal_actions[m][j] implies needed_machine[j]==m)
            if (jss_op_m(s.op[i]) == m_a) s.lb &= ~((((1u << jss_bs<KJ>()) | 1u)) << i);
    }
    // ONE inlined copy of the time advance serves the three callers: the raw hook (exactly one
    // advance), the no-op (:429-430, at least one) and the job branch (:469-470, zero or more)
    bool force = wait;
    uint32_t st;                                         // bit 0: some job is legal, bit 1: some event is pending
    for (;;) {
        st = __reduce_or_sync(JSS_FULL, ((s.lb & LM) != 0u ? 1u : 0u) | (s.tuam > 0 ? 2u : 0u));
        if (!(force || st == 2u)) break;                 // advance while nothing is legal and an event is pending
        holes += env_advance<KJ>(iv, s, lane);
        force = false;
        if (action == JSS_ACTION_ADVANCE) { raw_reward = -holes; return true; }   // heuristics / _is_done do NOT run
    }
    if (action == jss_J(iv) && !(st & 1u))
        s.flags |= JSS_FLAG_ERROR;                       // the reference raises here (queue ran empty)
    raw_reward = gain - holes;
    env_prioritize<KJ>(iv, s, lane);                     // :432 / :471
    const uint32_t ML = env_machine_legal<KJ>(s);
    const int nlegal = (int)__reduce_add_sync(JSS_FULL, (unsigned)__popc(s.lb & LM));
    const bool noop = env_check_no_op<KJ>(iv, s, lane, ML, nlegal, hz);   // :433 / :472
    s.flags &= ~(JSS_FLAG_NOOP_LEGAL | JSS_FLAG_DONE);
    if (noop) s.flags |= JSS_FLAG_NOOP_LEGAL;
    s.ep_steps += 1;
    s.ep_return += raw_reward;
    if (nlegal == 0) {                                   // _is_done (:649)
        s.flags |= JSS_FLAG_DONE;
        env_episode_end<KJ>(p, s, env, lane);
    }
    return true;
}

// ---- policies (JSSEnv/dispatching.py; README.md:58-60) ---------------------------------
template <int KJ, bool RANDOM_ONLY = false>
JSS_DEV int env_select_action(const InstView &iv, const EnvRegs<KJ> &s, int lane, int rule, int coin_mode,
                              uint32_t h, double cr_factor) {
    constexpr uint32_t LM = jss_legal_mask<KJ>();
    const uint32_t mine = (uint32_t)__popc(s.lb & LM);
    // inclusive prefix count of legal jobs over the lanes (ascending job index order)
    uint32_t incl = mine;
    int njobs;
    if (KJ == 1) {                                       // one job per lane: the prefix is a popcount of the ballot
        const uint32_t b = __ballot_sync(JSS_FULL, mine != 0u);
        incl = (uint32_t)__popc(b & ((2u << lane) - 1u));
        njobs = __popc(b);
    } else {
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const uint32_t o = __shfl_up_sync(JSS_FULL, incl, off);
            if (lane >= off) incl += o;
        }
        njobs = (int)__shfl_sync(JSS_FULL, incl, 31);
    }
    const bool noop = (s.flags & JSS_FLAG_NOOP_LEGAL) != 0u;
    if (s.flags & JSS_FLAG_DONE) return 0;               // ignored by step (auto-reset or frozen)
    if (njobs == 0) return noop ? jss_J(iv) : JSS_ACTION_SKIP;   // "only the no-op is legal" (e.g. :96-97)
    if (RANDOM_ONLY || rule == JSS_RULE_RANDOM) {
        // uniform over the set bits of action_mask, indexed in ascending action order
        const uint32_t r = jss_pick(h, (uint32_t)(njobs + (noop ? 1 : 0)));
        if ((int)r == njobs) return jss_J(iv);
        const uint32_t before = incl - mine;
        const bool own = r >= before && r < incl;
        int act = 0;
        uint32_t k = r - before;                         // k-th set slot of this lane (meaningful if `own`)
#pragma unroll
        for (int i = 0; i < KJ; i++) {
            const uint32_t bit = (s.lb >> i) & 1u;
            act = (bit && k == 0u) ? KJ * lane + i : act;
            k -= bit;
        }
        const uint32_t who = __ballot_sync(JSS_FULL, own);
        return __shfl_sync(JSS_FULL, act, __ffs((int)who) - 1);
    }
    int best;
    if (rule == JSS_RULE_CR) {                           // dispatching.py:365-408, float64 like Python
        double key = 1.0 / 0.0;
        int kj = 1 << 20;
#pragma unroll
        for (int i = 0; i < KJ; i++) {
            const int j = KJ * lane + i;
            if (s.lb & (1u << i)) {
                const double due = (double)iv.len[j] * cr_factor;                    // :357-360
                const int remaining = iv.rem[j * (jss_M(iv) + 1) + s.todo[i]];            // :387-388
                const double ratio = remaining > 0 ? (due - (double)s.t) / (double)remaining : 1.0 / 0.0;
                if (ratio < key) { key = ratio; kj = j; }                            // strict <, first index wins
            }
        }
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) {
            const double ok = __shfl_xor_sync(JSS_FULL, key, off);
            const int oj = __shfl_xor_sync(JSS_FULL, kj, off);
            if (ok < key || (ok == key && oj < kj)) { key = ok; kj = oj; }
        }
        best = kj;
    } else {
        // integer keys; composite (key << 8 | tie) so one REDUX picks value and first index
        const bool minimise = (rule == JSS_RULE_SPT || rule == JSS_RULE_LWR || rule == JSS_RULE_LOR);
        uint32_t comp = minimise ? 0xffffffffu : 0u;
#pragma unroll
        for (int i = 0; i < KJ; i++) {
            const int j = KJ * lane + i;
            if (s.lb & (1u << i)) {
                uint32_t key;
                if (rule == JSS_RULE_SPT) key = (uint32_t)jss_op_d(s.op[i]);                    // :105-108
                else if (rule == JSS_RULE_FIFO) key = (uint32_t)s.idle_last[i];                 // :146-148
                else if (rule == JSS_RULE_MWR || rule == JSS_RULE_LWR)
                    key = iv.rem[j * (jss_M(iv) + 1) + s.todo[i]];                                   // :188-191 / :231-234
                else key = (uint32_t)(jss_M(iv) - s.todo[i]);                                        // :273 / :314
                const uint32_t c = minimise ? ((key << 8) | (uint32_t)j) : ((key << 8) | (uint32_t)(255 - j));
                comp = minimise ? min(comp, c) : max(comp, c);
            }
        }
        comp = minimise ? __reduce_min_sync(JSS_FULL, comp) : __reduce_max_sync(JSS_FULL, comp);
        best = minimise ? (int)(comp & 255u) : 255 - (int)(comp & 255u);
    }
    if (noop && coin_mode == JSS_COIN_DEVICE && h < JSS_COIN_THRESHOLD) return jss_J(iv);   // e.g. :113-114
    return best;
}

// ---- canonical export / import (snapshot & restore; host attribute views) -------------
template <int KJ>
JSS_DEV void env_export(const JssParams &p, const InstView &iv, const EnvRegs<KJ> &s, int env, int lane) {
    const size_t jb = (size_t)env * p.jobs_max;
#pragma unroll
    for (int i = 0; i < KJ; i++) {
        const int j = KJ * lane + i;
        if (j < jss_J(iv)) {
            p.x_todo[jb + j] = s.todo[i]; p.x_tufco[jb + j] = s.tufco[i];
            p.x_idle_last[jb + j] = s.idle_last[i]; p.x_total_idle[jb + j] = s.total_idle[i];
            p.x_col4[jb + j] = s.col4[i];
            p.x_legal[jb + j] = (uint8_t)((s.lb >> i) & 1u);
            p.x_blocked[jb + j] = (uint8_t)((s.lb >> (jss_bs<KJ>() + i)) & 1u);
        }
    }
    if (lane < jss_M(iv)) p.x_tuam[(size_t)env * p.machines_max + lane] = s.tuam;
    if (lane == 0) {
        p.scalars[4 * (size_t)env + 2] = s.t;
        p.scalars[4 * (size_t)env + 3] = (int32_t)((s.flags << 8) | (s.flags & JSS_FLAG_DONE));
    }
}

template <int KJ>
JSS_DEV void env_import(const JssParams &p, const InstView &iv, EnvRegs<KJ> &s, int env, int lane) {
    const size_t jb = (size_t)env * p.jobs_max;
    s.lb = 0u;
#pragma unroll
    for (int i = 0; i < KJ; i++) {
        const int j = KJ * lane + i;
        const bool valid = j < jss_J(iv);
        s.todo[i] = valid ? p.x_todo[jb + j] : jss_M(iv);
        s.tufco[i] = valid ? p.x_tufco[jb + j] : 0;
        s.idle_last[i] = valid ? p.x_idle_last[jb + j] : 0;
        s.total_idle[i] = valid ? p.x_total_idle[jb + j] : 0;
        s.col4[i] = valid ? p.x_col4[jb + j] : 0;
        if (valid && p.x_legal[jb + j] != 0) s.lb |= 1u << i;
        if (valid && p.x_blocked[jb + j] != 0) s.lb |= (1u << jss_bs<KJ>()) << i;
    }
    s.tuam = lane < jss_M(iv) ? p.x_tuam[(size_t)env * p.machines_max + lane] : 0;
    s.t = p.scalars[4 * (size_t)env + 2];
    s.flags = (uint32_t)p.scalars[4 * (size_t)env + 3] >> 8;
    env_derive_ops<KJ>(iv, s, lane);
}

// ---- packed observation row (host-buffer path) ---------------------------------------------------------
// 10 bytes per job: w0 = legal | tufco << 1 | todo << 12 | col4 << 18, then idle_last and total_idle as 24-bit
// little-endian integers (the makespan bound J*M*2047 < 2^24).  Column 3 (total_perform) is derivable on the host
// from total_idle, todo, t and jobs_length.  jss_host_expand_obs() turns a row back into the exact real_obs floats.
template <int KJ>
JSS_DEV void env_pack(const JssLaunch &a, const InstView &iv, const EnvRegs<KJ> &s, int env, int lane, float *scratch) {
    uint16_t *st = reinterpret_cast<uint16_t *>(scratch);
    if (KJ * lane < jss_J(iv)) {
#pragma unroll
        for (int i = 0; i < KJ; i++) {
            const uint32_t w0 = ((s.lb >> i) & 1u) | ((uint32_t)s.tufco[i] << 1) | ((uint32_t)s.todo[i] << 12) |
                                ((uint32_t)s.col4[i] << 18);
            const uint32_t il = (uint32_t)s.idle_last[i], ti = (uint32_t)s.total_idle[i];
            uint16_t *r = st + 5 * (KJ * lane + i);
            r[0] = (uint16_t)w0; r[1] = (uint16_t)(w0 >> 16);
            r[2] = (uint16_t)il;                                      // bytes 4,5
            r[3] = (uint16_t)(((il >> 16) & 255u) | ((ti & 255u) << 8));   // byte 6 = idle[23:16], byte 7 = total[7:0]
            r[4] = (uint16_t)(ti >> 8);                               // bytes 8,9
        }
    }
    __syncwarp();
    uint4 *dst = reinterpret_cast<uint4 *>(a.wire + (size_t)env * a.wire_stride);
    const int n16 = (jss_J(iv) * 10 + 15) >> 4;
    for (int k = lane; k < n16; k += 32) dst[k] = reinterpret_cast<const uint4 *>(scratch)[k];
    __syncwarp();
}

// ---- CTA-level driver -----------------------------------------------------------------------
struct JssSmemLayout {
    // byte offsets from the start of dynamic shared memory, precomputed on the host so the kernels derive every
    // pointer with one add (each region 16-byte aligned): [SmInst][ops u16][len i32][rem u16][per-warp regions]
    int32_t off_len, off_rem, off_warp0, pad0_;
    int32_t warp_stride;    // bytes per warp region
    int32_t scratch_words;  // observation staging (7 floats per job slot), >= 32 words
    int32_t off_scratch;    // step kernels: [mbarrier 16 B][state-in block][scratch][state-out block]; else 0
    int32_t pad_;
};

struct JssCtaSmem {         // the CTA-shared part
    SmInst *si;
    uint16_t *ops;
    int32_t *len;
    uint16_t *rem;
};
JSS_DEV void jss_cta_carve(const JssSmemLayout &sl, char *sm, JssCtaSmem &c, InstView &iv) {
    c.si = reinterpret_cast<SmInst *>(sm);
    c.ops = reinterpret_cast<uint16_t *>(sm + sizeof(SmInst));
    c.len = reinterpret_cast<int32_t *>(sm + sl.off_len);
    c.rem = reinterpret_cast<uint16_t *>(sm + sl.off_rem);
    iv.ops = c.ops; iv.len = c.len; iv.rem = c.rem; iv.si = c.si; iv.staged = true; iv.Ju = iv.Mu = 0;
}

// refresh the uniform register copies of J / M from the staged instance (one packed shuffle)
JSS_DEV void jss_iv_shape(InstView &iv) {
    const uint32_t jm = jss_uniform((uint32_t)iv.si->J | ((uint32_t)iv.si->M << 16));
    iv.Ju = (int)(jm & 0xffffu); iv.Mu = (int)(jm >> 16);
}

#define JSS_STAGE_OPS 1     // ops + jobs_length
#define JSS_STAGE_REM 2     // suffix sums (rules MWR / LWR / CR)
#define JSS_STAGE_ALL 3
// the rules that read the suffix sums; the host sizes the shared-memory layout with the same predicate
JSS_DEV bool jss_rule_wants_rem(int rule) { return rule == JSS_RULE_MWR || rule == JSS_RULE_LWR || rule == JSS_RULE_CR; }

JSS_DEV void jss_fill_sminst(const JssInstDesc &d, SmInst *si) {
    si->J = d.J; si->M = d.M; si->max_time_op = d.max_time_op; si->max_time_jobs = d.max_time_jobs;
    si->sum_op = d.sum_op;
    si->f_mto = (float)d.max_time_op; si->f_mtj = (float)d.max_time_jobs; si->f_sop = (float)d.sum_op;
    si->f_M = (float)d.M;
    si->r_mto = d.r_mto; si->r_mtj = d.r_mtj; si->r_sop = d.r_sop; si->r_M = d.r_M;
    // per-lane slices are whole vectors: J rounded up to 4 (to 8 for the 8-jobs-per-lane class, which also keeps 16 bits per lane)
    si->Jcap = d.J > 128 ? ((d.J + 7) & ~7) : ((d.J + 3) & ~3); si->Mcap = (d.M + 3) & ~3;
    si->block_words = 5 * si->Jcap + si->Mcap + (d.J > 128 ? 16 : 8) + 4;
    si->n14[0] = si->n14[1] = -si->f_mto; si->r14[0] = si->r14[1] = d.r_mto;
    si->n23[0] = -si->f_M; si->n23[1] = -si->f_mtj; si->r23[0] = d.r_M; si->r23[1] = d.r_mtj;
    si->n56[0] = si->n56[1] = -si->f_sop; si->r56[0] = si->r56[1] = d.r_sop;
}

JSS_DEV void jss_stage_instance(const JssParams &p, const JssInstDesc &d, const JssCtaSmem &c, int what) {
    const int tid = threadIdx.x, nt = blockDim.x;
    if (tid == 0) jss_fill_sminst(d, c.si);
    // pools are padded so whole uint4 copies stay in-bounds
    if (what & JSS_STAGE_OPS) {
        {
            const uint4 *src = reinterpret_cast<const uint4 *>(p.ops_pool + d.ops_off);
            uint4 *dst = reinterpret_cast<uint4 *>(c.ops);
            const int n = (d.J * d.M + 7) >> 3;
            for (int k = tid; k < n; k += nt) dst[k] = src[k];
        }
        {
            const uint4 *src = reinterpret_cast<const uint4 *>(p.len_pool + d.len_off);
            uint4 *dst = reinterpret_cast<uint4 *>(c.len);
            const int n = (d.J + 3) >> 2;
            for (int k = tid; k < n; k += nt) dst[k] = src[k];
        }
    }
    if (what & JSS_STAGE_REM) {
        const uint4 *src = reinterpret_cast<const uint4 *>(p.rem_pool + d.rem_off);
        uint4 *dst = reinterpret_cast<uint4 *>(c.rem);
        const int n = (d.J * (d.M + 1) + 7) >> 3;
        for (int k = tid; k < n; k += nt) dst[k] = src[k];
    }
}

template <int KJ, bool BULK = false>
JSS_DEV void env_emit_all(const JssParams &p, const InstView &iv, const EnvRegs<KJ> &s, int env, int lane,
                          float *scratch, int raw, jss_saddr_t scratch_sa = jss_saddr_t(), void *st_dst = nullptr,
                          jss_saddr_t st_sa = jss_saddr_t(), uint32_t st_bytes = 0u) {
    const JssOut out = jss_out_default(p);
    env_emit_obs<KJ, BULK>(p, out, iv, s, env, lane, scratch, scratch_sa, st_dst, st_sa, st_bytes);
    env_emit_mask<KJ>(p, out, iv, s, env, lane, (s.flags & JSS_FLAG_NOOP_LEGAL) != 0u);
    env_emit_scalars<KJ>(out, iv, s, env, lane, raw);
}

// ---- generator mode: draw instance k of an env (jss_gen.h) --------------------------------------------------
// Lane l generates the rows of its KJ jobs; the three scalars are warp reductions, the reciprocals IEEE divisions, so the
// desc and tables equal what jss_load_instances builds from the same arrays.  Writes the env's tables in HBM, the same
// [desc][ops][len] unit into the warp's shared-memory table buffer `tb` (if given), and the warp's SmInst.
template <int KJ>
JSS_DEV void jss_gen_draw(const JssGenParams &g, uint64_t genv, int env, int k, int lane, char *tb, SmInst *si) {
    const int J = g.J, M = g.M;
    char *tg = g.tables + (size_t)env * g.tbl_bytes;
    uint16_t *ops = reinterpret_cast<uint16_t *>(tg + JSS_GEN_HDR_BYTES);
    int32_t *len = reinterpret_cast<int32_t *>(tg + JSS_GEN_HDR_BYTES + g.ops_bytes);
    uint16_t *rem = g.rem + (size_t)env * g.rem_elems;
    int32_t mto = 0, mtj = 0, sop = 0;
#pragma unroll
    for (int i = 0; i < KJ; i++) {
        const int j = KJ * lane + i;
        if (j < J) {
            uint8_t mach[JSS_MAX_MACHINES];
            int32_t dur[JSS_MAX_MACHINES];
            jss_gen_row(g.seed, genv, (uint64_t)k, j, M, g.dmin, g.dmax, mach, dur);
            int32_t mx = 0;
            const int32_t l = jss_pack_job_row(mach, dur, M, ops + j * M, rem + j * (M + 1), &mx);
            len[j] = l;
            if (tb) {
                uint16_t *so = reinterpret_cast<uint16_t *>(tb + JSS_GEN_HDR_BYTES) + j * M;
                for (int q = 0; q < M; q++) so[q] = ops[j * M + q];
                reinterpret_cast<int32_t *>(tb + JSS_GEN_HDR_BYTES + g.ops_bytes)[j] = l;
            }
            mto = max(mto, mx); mtj = max(mtj, l); sop += l;
        }
    }
    mto = (int32_t)__reduce_max_sync(JSS_FULL, (unsigned)mto);
    mtj = (int32_t)__reduce_max_sync(JSS_FULL, (unsigned)mtj);
    sop = (int32_t)__reduce_add_sync(JSS_FULL, (unsigned)sop);
    if (lane == 0) {
        const JssInstDesc d = jss_inst_desc(J, M, mto, mtj, sop);
        *reinterpret_cast<JssInstDesc *>(tg) = d;
        if (tb) *reinterpret_cast<JssInstDesc *>(tb) = d;
        jss_fill_sminst(d, si);
        g.index[env] = k;
    }
    // the tables were written through the generic proxy; the step kernel reads them with bulk copies (async proxy)
    jss_fence_async_global();
    __syncwarp();
}

// GEN: generator mode (jss_gen_env_kernel): `iv` points at the env's own tables, iv.si at the warp's own SmInst, and every
// reset -- explicit, or the auto-reset inside a rollout -- first draws the env's next instance.
template <int KJ, int MODE, bool GEN = false>
JSS_DEV void jss_process_env(const JssParams &p, const JssLaunch &a, const InstView &iv, int env, int lane,
                             float *scratch, const JssGenParams *g = nullptr) {
    EnvRegs<KJ> s;
    // MODE is a compile-time kernel variant (the hot step kernel carries no policy /
    // rollout / export code); JSS_MODE_RESET instantiates the rarely used rest
    const int mode = (MODE == JSS_MODE_RESET) ? a.mode : MODE;
    int *hz = reinterpret_cast<int *>(scratch);
    if (mode == JSS_MODE_RESET) {
        if (a.env_mask && a.env_mask[env] == 0) return;
        if (GEN) jss_gen_draw<KJ>(*g, p.env_id_base + (uint64_t)env, env, g->index[env] + 1, lane, nullptr, const_cast<SmInst *>(iv.si));
        env_reset_regs<KJ>(iv, s, lane);
        if (p.solution) {
            int32_t *sol = p.solution + (size_t)env * p.jobs_max * p.machines_max;
            for (int k = lane; k < p.jobs_max * p.machines_max; k += 32) sol[k] = -1;
        }
        env_store<KJ>(p, iv, env, lane, s);
        env_emit_all<KJ>(p, iv, s, env, lane, scratch, 0);
        return;
    }
    if (mode == JSS_MODE_IMPORT) {
        if (a.env_mask && a.env_mask[env] == 0) return;
        env_import<KJ>(p, iv, s, env, lane);
        s.ep_steps = 0; s.ep_return = 0;
        env_store<KJ>(p, iv, env, lane, s);
        env_emit_obs<KJ>(p, jss_out_default(p), iv, s, env, lane, scratch);
        env_emit_mask<KJ>(p, jss_out_default(p), iv, s, env, lane, (s.flags & JSS_FLAG_NOOP_LEGAL) != 0u);
        if (lane == 0) p.scalars[4 * (size_t)env + 3] = (int32_t)((s.flags << 8) | (s.flags & JSS_FLAG_DONE));
        return;
    }
    const uint64_t genv = p.env_id_base + (uint64_t)env;
    if (mode == JSS_MODE_POLICY) env_load_for_policy<KJ>(p, iv, env, lane, s, a.rule);
    else env_load<KJ>(p, iv, env, lane, s);
    s.flags = jss_uniform(s.flags);                      // one word read by every lane (see jss_uniform)
    if (mode == JSS_MODE_EXPORT) { env_export<KJ>(p, iv, s, env, lane); return; }
    if (mode == JSS_MODE_PACK) { env_pack<KJ>(a, iv, s, env, lane, scratch); return; }
    if (mode == JSS_MODE_POLICY) {
        const uint32_t h = jss_hash3(a.seed, genv, a.step_index);
        const int act = env_select_action<KJ>(iv, s, lane, a.rule, a.coin_mode, h, a.cr_factor);
        if (lane == 0) a.actions_out[env] = act;
        return;
    }
    if (mode == JSS_MODE_STEP) {
        const int action = jss_uniform(a.actions[env]);
        int raw = 0;
        const uint32_t flags_in = s.flags;
        const bool changed = env_step<KJ>(p, iv, s, env, lane, action, raw, hz);
        s.flags = jss_uniform(s.flags);
        if (changed) {
            env_store<KJ>(p, iv, env, lane, s);
            env_emit_all<KJ>(p, iv, s, env, lane, scratch, raw);
        } else if (s.flags != flags_in) {                // only the sticky error bit changed
            if (lane == 0) {
                p.state[(size_t)p.hdr_off16[env] * 4 + JSS_HDR_FLAGS] = (int32_t)s.flags;
                reinterpret_cast<int4 *>(p.scalars)[env] =
                    make_int4(0, 0, s.t, (int)((s.flags << 8) | (s.flags & JSS_FLAG_DONE)));
            }
        }
        if (a.export_after) env_export<KJ>(p, iv, s, env, lane);   // single-env facade: one launch per transition
        return;
    }
    // JSS_MODE_ROLLOUT: n_steps x (policy -> step) with the state held in registers.
    // Trajectory recording (a.traj_obs != NULL): step k of this env writes its observation / mask / scalar record (and
    // the action that led to it) into slot k * n_envs + env of the caller's [n_steps][N][...] buffers -- the emit helpers
    // index their outputs by env only, so a shifted index and other base pointers are all it takes (ONE loop body).
    const bool record = a.traj_obs != nullptr;
    const JssOut out = record ? JssOut{a.traj_obs, a.traj_mask, a.traj_scalars} : jss_out_default(p);
    bool dirty = false;
    int raw = 0;
    for (int k = 0; k < a.n_steps; k++) {
        const uint32_t h = jss_hash3(a.seed, genv, a.step_index + (uint64_t)k);
        const int act = jss_uniform(env_select_action<KJ>(iv, s, lane, a.rule, a.coin_mode, h, a.cr_factor));
        if (GEN && (s.flags & JSS_FLAG_DONE) && (p.create_flags & JSS_CREATE_AUTO_RESET))   // env_step resets it now
            jss_gen_draw<KJ>(*g, genv, env, g->index[env] + 1, lane, nullptr, const_cast<SmInst *>(iv.si));
        int r = 0;
        const bool changed = env_step<KJ>(p, iv, s, env, lane, act, r, hz);
        s.flags = jss_uniform(s.flags);
        if (changed) { raw = r; dirty = true; }
        if (record || (changed && a.write_obs)) {
            const int slot = record ? k * p.n_envs + env : env;
            if (record && a.traj_actions && lane == 0) a.traj_actions[slot] = act;
            env_emit_obs<KJ>(p, out, iv, s, slot, lane, scratch);
            env_emit_mask<KJ>(p, out, iv, s, slot, lane, (s.flags & JSS_FLAG_NOOP_LEGAL) != 0u);
            env_emit_scalars<KJ>(out, iv, s, slot, lane, changed ? r : 0);
        }
    }
    if (dirty) {
        env_store<KJ>(p, iv, env, lane, s);
        if (!a.write_obs || record) env_emit_all<KJ>(p, iv, s, env, lane, scratch, raw);
    }
}

JSS_DEV void jss_tile_desc(const JssParams &p, int tile, int &first, int &inst, int &count) {
    if (p.uniform_inst >= 0) {           // one instance, identity order: no descriptor loads
        first = tile * JSS_WARPS_PER_CTA;
        inst = p.uniform_inst;
        count = min(JSS_WARPS_PER_CTA, p.n_envs - first);
    } else {
        const JssTile td = p.tiles[tile];
        first = td.first; inst = td.inst_count >> 8; count = td.inst_count & 255;
    }
}

#ifndef JSS_MIN_CTAS
#define JSS_MIN_CTAS 3   // 78 registers, no spills -> 3 CTAs = 24 warps per SM (sweeps in profiles/)
#endif
#ifndef JSS_MIN_CTAS_SMALL
#define JSS_MIN_CTAS_SMALL 4   // uniform batches with <= 32 jobs (KJ = 1) are latency-bound: 4 CTAs = 32 warps per SM at 64 registers
#endif                         // (measured: 15x15 .. 30x20 shapes -4 %, ta01 N = 4096 8.1 -> 6.7 us per step; no gain for KJ = 2)

template <int KJ, int MODE>
__global__ void __launch_bounds__(JSS_WARPS_PER_CTA * 32, 1)
jss_env_kernel(const JssParams p, const JssLaunch a, const JssSmemLayout sl) {
    JSS_SMEM_DECL(jss_smem);
    char *sm = reinterpret_cast<char *>(jss_smem);
    JssCtaSmem c;
    InstView iv;
    jss_cta_carve(sl, sm, c, iv);
    const int warp = jss_warp_index(), lane = threadIdx.x & 31;
    float *scratch = reinterpret_cast<float *>(sm + sl.off_warp0 + warp * sl.warp_stride);
    // what the mode reads: the masked-uniform sampler looks at no instance table at all (only J); the other policies
    // at ops / len (+ suffix sums for MWR / LWR / CR); everything that steps needs all tables
    int what = JSS_STAGE_OPS;
    if (MODE == JSS_MODE_ROLLOUT) what = JSS_STAGE_ALL;
    if (MODE == JSS_MODE_POLICY)
        what = a.rule == JSS_RULE_RANDOM ? 0 : jss_rule_wants_rem(a.rule) ? JSS_STAGE_ALL : JSS_STAGE_OPS;
    int staged = -1;
    for (int tile = a.tile_begin + (int)blockIdx.x; tile < a.tile_end; tile += (int)gridDim.x) {
        int first, inst, count;
        jss_tile_desc(p, tile, first, inst, count);
        first = jss_uniform(first); inst = jss_uniform(inst); count = jss_uniform(count);
        if (inst != staged) {                            // CTA-uniform
            __syncthreads();
            jss_stage_instance(p, p.inst[inst], c, what);
            staged = inst;
            __syncthreads();
        }
        jss_iv_shape(iv);
        if (warp < count)
            jss_process_env<KJ, MODE>(p, a, iv, p.uniform_inst >= 0 ? first + warp : jss_uniform(p.order[first + warp]),
                                      lane, scratch);
    }
}

// Generator mode, everything but the step (reset, policy, rollout, export): uniform geometry and identity order like a
// uniform batch, but each warp points its InstView at its own env's tables in HBM and keeps its own SmInst in shared
// memory -- no CTA barrier.  Per warp: [SmInst][scratch], g.warp_stride bytes.
template <int KJ, int MODE>
__global__ void __launch_bounds__(JSS_WARPS_PER_CTA * 32, 1)
jss_gen_env_kernel(const JssParams p, const JssLaunch a, const JssGenParams g) {
    JSS_SMEM_DECL(jss_smem);
    const int warp = jss_warp_index(), lane = threadIdx.x & 31;
    char *wb = reinterpret_cast<char *>(jss_smem) + warp * g.warp_stride;
    SmInst *si = reinterpret_cast<SmInst *>(wb);
    float *scratch = reinterpret_cast<float *>(wb + sizeof(SmInst));
    InstView iv;
    iv.si = si; iv.staged = true; iv.Ju = g.J; iv.Mu = g.M;
    for (int tile = a.tile_begin + (int)blockIdx.x; tile < a.tile_end; tile += (int)gridDim.x) {
        const int env = tile * JSS_WARPS_PER_CTA + warp;
        if (env >= p.n_envs) break;
        const char *tg = g.tables + (size_t)env * g.tbl_bytes;
        iv.ops = reinterpret_cast<const uint16_t *>(tg + JSS_GEN_HDR_BYTES);
        iv.len = reinterpret_cast<const int32_t *>(tg + JSS_GEN_HDR_BYTES + g.ops_bytes);
        iv.rem = g.rem + (size_t)env * g.rem_elems;
        if (lane == 0) jss_fill_sminst(*reinterpret_cast<const JssInstDesc *>(tg), si);
        __syncwarp();
        jss_process_env<KJ, MODE, true>(p, a, iv, env, lane, scratch, &g);
        __syncwarp();                                    // every lane is done with si before the next env refills it
    }
}

// ---- programmatic dependent launch (PDL) -------------------------------------------------------
// The step kernels are launched with cudaLaunchAttributeProgrammaticStreamSerialization: the NEXT
// launch's CTAs may become resident (and run their prologue: shared-memory carve-up, mbarrier init,
// staging of the read-only instance tables) while this launch drains; jss_pdl_wait() blocks them until
// every memory operation of the preceding grid is visible, so nothing mutable is touched before it.
#ifndef JSS_EMU
JSS_DEV void jss_pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
JSS_DEV void jss_pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
#else
JSS_DEV void jss_pdl_launch_dependents() {}
JSS_DEV void jss_pdl_wait() {}
#endif

// ---- the hot kernels: fused step with TMA prefetch ---------------------------------------------
// Persistent CTAs (grid = SMs x resident CTAs), one warp per env of a tile.  Per warp in shared
// memory: an mbarrier, a state-block buffer that receives the NEXT env's block by cp.async.bulk
// while the current env is simulated, and the staging buffers (new state block, observation rows)
// that leave by bulk store.
// SAMPLE = 1 / 2 additionally picks every env's NEXT action (masked-uniform sampler / any dispatching
// rule) from the freshly computed state, so a policy-driven loop is one launch per step.
struct JssWarpSmem {        // per-warp shared-memory regions of the step kernels
    int32_t *state_in, *state_out;
    float *scratch;
    jss_saddr_t mbar, state_sa, scratch_sa, state_out_sa;
};

// env handled by `warp` in `tile` (-1: none) and where its state block lives (16-byte units)
template <bool UNI>
JSS_DEV int jss_tile_env(const JssParams &p, const JssLaunch &a, int tile, int tile_end, int warp, int lane,
                         uint32_t &off16, uint32_t &blk16) {
    if (UNI) {                           // env = 8 * tile + warp, block = env * block_words: nothing to load
        const int e = tile * JSS_WARPS_PER_CTA + warp;
        blk16 = (uint32_t)a.uni.block_words >> 2;
        off16 = (uint32_t)e * blk16;
        return (tile < tile_end && e < p.n_envs) ? e : -1;
    }
    if (tile >= tile_end) return -1;
    const int4 td = *reinterpret_cast<const int4 *>(p.tiles + tile);     // JssTile, one 16-byte load
    if (warp >= (td.y & 255)) return -1;
    blk16 = (uint32_t)td.w;
    off16 = (uint32_t)td.z + (uint32_t)warp * blk16;
    return p.order[td.x + warp];
}

// where the state block of warp `warp` of `tile` lives (16-byte units); recomputed after the step instead of
// being carried in registers across it
template <bool UNI>
JSS_DEV void jss_tile_state(const JssParams &p, const SmInst *uni, int tile, int warp, int env, uint32_t &off16,
                            uint32_t &blk16) {
    if (UNI) {
        blk16 = (uint32_t)uni->block_words >> 2;
        off16 = (uint32_t)env * blk16;
    } else {
        const int4 td = *reinterpret_cast<const int4 *>(p.tiles + tile);
        blk16 = (uint32_t)td.w;
        off16 = (uint32_t)td.z + (uint32_t)warp * blk16;
    }
}

// tiles tile, tile + tile_step, ... < tile_end of ONE lane class through the prefetch pipeline
template <int KJ, int SAMPLE, bool UNI>
JSS_DEV void jss_step_tiles(const JssParams &p, const JssLaunch &a, const JssSmemLayout &sl, InstView &iv,
                            const JssCtaSmem &c, const JssWarpSmem &w, int warp, int lane, int tile, int tile_end,
                            int tile_step, int &staged, uint32_t &phase) {
    int env_next, act_next = 0;
    {
        uint32_t off16, blk16;
        env_next = jss_tile_env<UNI>(p, a, tile, tile_end, warp, lane, off16, blk16);
        if (env_next >= 0) {
            if (lane == 0) jss_bulk_load(w.state_sa, p.state + (size_t)off16 * 4, blk16 * 16u, w.mbar);
            act_next = a.actions[env_next];
        }
    }
    for (; tile < tile_end; tile += tile_step) {
        if (!UNI) {
            const int inst = p.tiles[tile].inst_count >> 8;
            if (inst != staged) {                        // CTA-uniform
                __syncthreads();
                jss_stage_instance(p, p.inst[inst], c, (SAMPLE == 2 && jss_rule_wants_rem(a.rule)) ? JSS_STAGE_ALL : JSS_STAGE_OPS);
                staged = inst;
                __syncthreads();
            }
            jss_iv_shape(iv);
        }
        const int env = UNI ? env_next : jss_uniform(env_next), action = act_next;
        EnvRegs<KJ> s;
        if (env >= 0) {
            jss_mbar_wait(w.mbar, phase);                // this env's block has landed in shared memory
            phase ^= 1u;
            env_load_from<KJ>(p, iv, w.state_in, lane, s);
            __syncwarp();                                // every lane has read the buffer
        }
        {   // prefetch the next env's block + action
            uint32_t off16, blk16;
            env_next = jss_tile_env<UNI>(p, a, tile + tile_step, tile_end, warp, lane, off16, blk16);
            if (env_next >= 0) {
                if (lane == 0) jss_bulk_load(w.state_sa, p.state + (size_t)off16 * 4, blk16 * 16u, w.mbar);
                act_next = a.actions[env_next];
            }
        }
        if (env < 0) continue;
        int raw = 0;
        // the previous env's observation must have left the staging buffer (also aliased by hz)
        if (lane == 0) jss_bulk_store_wait_read();
        __syncwarp();
        // every lane holds the same flags word (one address, loaded by all lanes): say so -- ptxas already sees that
        // for the action and the time, a shuffle of those is folded away
        if (jss_hint_flags<KJ, UNI>()) s.flags = jss_uniform(s.flags);
        const uint32_t flags_in = s.flags;
        const bool changed = env_step<KJ>(p, iv, s, env, lane, action, raw, reinterpret_cast<int *>(w.scratch));
        if (jss_hint_flags<KJ, UNI>()) s.flags = jss_uniform(s.flags);   // the no-op test returns from inside lane-dependent code
        if (SAMPLE) {
            const uint32_t h = jss_hash_env(a.hash_key, p.env_id_base + (uint64_t)env);   // == jss_hash3(seed, genv, step_index)
            const int nxt = env_select_action<KJ, SAMPLE == 1>(iv, s, lane, a.rule, a.coin_mode, h, a.cr_factor);
            if (lane == 0) a.actions_out[env] = nxt;
        }
        if (changed) {
            // new state -> shared staging -> one bulk store (every word of the block is rewritten)
            env_store_to<KJ>(p, iv, w.state_out, lane, s);
            uint32_t off16, blk16;
            jss_tile_state<UNI>(p, &a.uni, tile, warp, env, off16, blk16);
            env_emit_all<KJ, true>(p, iv, s, env, lane, w.scratch, raw, w.scratch_sa,
                                   p.state + (size_t)off16 * 4, w.state_out_sa, blk16 * 16u);
        } else if (s.flags != flags_in) {                // only the sticky error bit changed
            if (lane == 0) {
                p.state[(size_t)p.hdr_off16[env] * 4 + JSS_HDR_FLAGS] = (int32_t)s.flags;
                reinterpret_cast<int4 *>(p.scalars)[env] =
                    make_int4(0, 0, s.t, (int)((s.flags << 8) | (s.flags & JSS_FLAG_DONE)));
            }
        }
    }
}

JSS_DEV void jss_step_carve(const JssSmemLayout &sl, char *sm, int warp, JssWarpSmem &w) {
    int woff = sl.off_warp0 + warp * sl.warp_stride;
#if !defined(JSS_NO_OPAQUE_WBASE) && !defined(JSS_EMU)
    // keep the warp's region offset in ONE register instead of letting the optimiser recompute it from threadIdx
    // (S2R + shift + multiply-add) at every use: -1 % on the uniform ta80 step (94.0 -> 93.2 us)
    asm volatile("" : "+r"(woff));
#endif
    char *wbase = sm + woff;
    w.state_in = reinterpret_cast<int32_t *>(wbase + 16);
    w.scratch = reinterpret_cast<float *>(wbase + sl.off_scratch);
    w.mbar = jss_saddr(sm) + woff;   // shared-space addresses
    w.state_sa = w.mbar + 16;
    w.scratch_sa = w.mbar + sl.off_scratch;
    // state-out staging sits right behind the observation staging (both leave by bulk store)
    w.state_out = reinterpret_cast<int32_t *>(w.scratch + sl.scratch_words);
    w.state_out_sa = w.scratch_sa + sl.scratch_words * 4;
}

// Uniform batch (every env runs the same instance): static strided tiles, the per-instance scalars are
// read from the kernel parameters (constant-bank operands), no CTA barrier after the first staging.
template <int KJ, int SAMPLE>
__global__ void __launch_bounds__(JSS_WARPS_PER_CTA * 32, KJ == 1 ? JSS_MIN_CTAS_SMALL : (KJ == 8 ? 1 : JSS_MIN_CTAS))
jss_step_kernel(const JssParams p, const JssLaunch a, const JssSmemLayout sl) {
    JSS_SMEM_DECL(jss_smem);
    char *sm = reinterpret_cast<char *>(jss_smem);
    JssCtaSmem c;
    InstView iv;
    jss_cta_carve(sl, sm, c, iv);
    iv.si = &a.uni; iv.staged = false;
    const int warp = jss_warp_index(), lane = threadIdx.x & 31;
    JssWarpSmem w;
    jss_step_carve(sl, sm, warp, w);
    if (lane == 0) jss_mbar_init(w.mbar);
    jss_pdl_launch_dependents();
    // prologue on read-only data (overlaps the tail of the previous launch under PDL)
    jss_stage_instance(p, p.inst[p.uniform_inst], c, (SAMPLE == 2 && jss_rule_wants_rem(a.rule)) ? JSS_STAGE_ALL : JSS_STAGE_OPS);
    __syncthreads();
    jss_pdl_wait();
    int staged = p.uniform_inst;
    uint32_t phase = 0;
    // Static strided tiles; the env after the current one is known one iteration ahead, which is what
    // the TMA prefetch needs.
    jss_step_tiles<KJ, SAMPLE, true>(p, a, sl, iv, c, w, warp, lane, a.tile_begin + (int)blockIdx.x, a.tile_end,
                                     (int)gridDim.x, staged, phase);
    if (lane == 0) jss_bulk_store_wait_all();            // shared memory must outlive the bulk reads
}

// Mixed batch: ONE persistent launch covers the three lane classes.  Every CTA gets an equal slice of EVERY class
// (tile counts differ by at most one per class, the extras dithered across CTAs), so the launch is balanced without a
// cost model, and walks them class by class -- three complete loops in sequence, so each lane class keeps the register
// allocation of its stand-alone kernel.  All CTAs start with the 100-job class and move on at about the same time:
// the CTAs that share an SM mostly execute the same 20-35 KB loop body (the three together are 67-86 KB, more than
// the instruction cache holds).  Instance tables are re-staged only when the instance changes.
template <int SAMPLE, bool BIG>   // BIG: the batch contains instances with 129..256 jobs (a fourth, 8-jobs-per-lane body)
__global__ void __launch_bounds__(JSS_WARPS_PER_CTA * 32, BIG ? 1 : JSS_MIN_CTAS)
jss_step_mixed_kernel(const JssParams p, const JssLaunch a, const JssSmemLayout sl) {
    JSS_SMEM_DECL(jss_smem);
    char *sm = reinterpret_cast<char *>(jss_smem);
    JssCtaSmem c;
    InstView iv;
    jss_cta_carve(sl, sm, c, iv);
    const int warp = jss_warp_index(), lane = threadIdx.x & 31;
    JssWarpSmem w;
    jss_step_carve(sl, sm, warp, w);
    if (lane == 0) jss_mbar_init(w.mbar);
    jss_pdl_launch_dependents();
    const int4 r0 = reinterpret_cast<const int4 *>(p.cta_ranges + blockIdx.x)[0];   // [a4, b4) [a2, b2)
    const int4 r1 = reinterpret_cast<const int4 *>(p.cta_ranges + blockIdx.x)[1];   // [a1, b1) [a8, b8)
    jss_pdl_wait();
    int staged = -1;
    uint32_t phase = 0;
    if (BIG) jss_step_tiles<8, SAMPLE, false>(p, a, sl, iv, c, w, warp, lane, r1.z, r1.w, 1, staged, phase);   // 129..256 jobs
    jss_step_tiles<4, SAMPLE, false>(p, a, sl, iv, c, w, warp, lane, r0.x, r0.y, 1, staged, phase);
    jss_step_tiles<2, SAMPLE, false>(p, a, sl, iv, c, w, warp, lane, r0.z, r0.w, 1, staged, phase);
    jss_step_tiles<1, SAMPLE, false>(p, a, sl, iv, c, w, warp, lane, r1.x, r1.y, 1, staged, phase);
    if (lane == 0) jss_bulk_store_wait_all();            // shared memory must outlive the bulk reads
}

// Generator mode (every env has its own instance): the structure of the uniform step kernel -- persistent CTAs, static
// strided envs, the next env's state block prefetched by TMA -- plus, in the same bulk batch on the same mbarrier, that
// env's [desc][ops][len] table unit into the other half of a double-buffered per-warp table buffer (the current env reads
// its half for the whole step).  The suffix sums (only MWR / LWR / CR read them) are read through L1 from HBM.
// A done env that auto-resets draws its next instance here, before env_step's reset path runs.
// Per warp, behind the step region of jss_step_carve: [SmInst][table unit 0][table unit 1].
#ifndef JSS_GEN_STEP_WARPS
#define JSS_GEN_STEP_WARPS 4   // 4-warp CTAs: the double-buffered tables of 100x20 envs take 16 KB of shared memory per warp
#endif
struct JssGenStepArgs {      // shared-memory layout + generator-mode tables of the step kernel
    JssSmemLayout sl;
    JssGenParams g;
};
template <int KJ, int SAMPLE>
__global__ void __launch_bounds__(JSS_GEN_STEP_WARPS * 32, KJ == 1 ? 2 * JSS_MIN_CTAS_SMALL : 2 * JSS_MIN_CTAS)
jss_gen_step_kernel(const JssParams p, const JssLaunch a, const JssGenStepArgs ga) {
    const JssSmemLayout &sl = ga.sl;
    const JssGenParams &g = ga.g;
    JSS_SMEM_DECL(jss_smem);
    char *sm = reinterpret_cast<char *>(jss_smem);
    const int warp = jss_warp_index(), lane = threadIdx.x & 31;
    JssWarpSmem w;
    jss_step_carve(sl, sm, warp, w);
    char *wg = sm + sl.off_warp0 + warp * sl.warp_stride + g.off_gen;
    SmInst *si = reinterpret_cast<SmInst *>(wg);
    char *tb0 = wg + sizeof(SmInst);
    const jss_saddr_t tb0_sa = w.mbar + (uint32_t)(g.off_gen + (int)sizeof(SmInst));
    if (lane == 0) jss_mbar_init(w.mbar);
    jss_pdl_launch_dependents();
    __syncwarp();
    jss_pdl_wait();
    InstView iv;
    iv.si = si; iv.staged = true; iv.Ju = g.J; iv.Mu = g.M;
    const uint32_t blk16 = (uint32_t)a.uni.block_words >> 2, tbl_bytes = (uint32_t)g.tbl_bytes;
    const int env_step_stride = (int)gridDim.x * JSS_GEN_STEP_WARPS;
    uint32_t phase = 0, buf = 0;
    int env_next = (int)blockIdx.x * JSS_GEN_STEP_WARPS + warp, act_next = 0;
    if (env_next < p.n_envs) {
        if (lane == 0) {
            jss_mbar_expect_tx(w.mbar, blk16 * 16u + tbl_bytes);
            jss_bulk_copy(w.state_sa, p.state + (size_t)env_next * blk16 * 4, blk16 * 16u, w.mbar);
            jss_bulk_copy(tb0_sa, g.tables + (size_t)env_next * tbl_bytes, tbl_bytes, w.mbar);
        }
        act_next = a.actions[env_next];
    }
    while (env_next < p.n_envs) {
        const int env = env_next, action = act_next;
        char *tb = tb0 + buf * tbl_bytes;
        jss_mbar_wait(w.mbar, phase);                    // this env's state block and tables have landed
        phase ^= 1u;
        iv.ops = reinterpret_cast<const uint16_t *>(tb + JSS_GEN_HDR_BYTES);
        iv.len = reinterpret_cast<const int32_t *>(tb + JSS_GEN_HDR_BYTES + g.ops_bytes);
        iv.rem = g.rem + (size_t)env * g.rem_elems;
        if (lane == 0) jss_fill_sminst(*reinterpret_cast<const JssInstDesc *>(tb), si);
        __syncwarp();
        EnvRegs<KJ> s;
        env_load_from<KJ>(p, iv, w.state_in, lane, s);
        __syncwarp();                                    // every lane has read the state buffer
        env_next = env + env_step_stride;
        // the warp's generic-proxy accesses of the buffers the prefetch overwrites (the state buffer just read, the other
        // table half, which the generator may have written two envs ago) must be ordered before its async-proxy writes:
        // without this fence, 65 536-env runs of 100x20 saw torn tables after auto-resets (observations outside [0, 1])
        jss_fence_async_smem();
        __syncwarp();
        if (env_next < p.n_envs) {                       // prefetch the next env's block + tables + action
            if (lane == 0) {
                jss_mbar_expect_tx(w.mbar, blk16 * 16u + tbl_bytes);
                jss_bulk_copy(w.state_sa, p.state + (size_t)env_next * blk16 * 4, blk16 * 16u, w.mbar);
                jss_bulk_copy(tb0_sa + (buf ^ 1u) * tbl_bytes, g.tables + (size_t)env_next * tbl_bytes, tbl_bytes, w.mbar);
            }
            act_next = a.actions[env_next];
        }
        s.flags = jss_uniform(s.flags);
        if ((s.flags & JSS_FLAG_DONE) && action != JSS_ACTION_SKIP && (p.create_flags & JSS_CREATE_AUTO_RESET))
            jss_gen_draw<KJ>(g, p.env_id_base + (uint64_t)env, env, g.index[env] + 1, lane, tb, si);
        int raw = 0;
        // the previous env's observation must have left the staging buffer (also aliased by hz)
        if (lane == 0) jss_bulk_store_wait_read();
        __syncwarp();
        const uint32_t flags_in = s.flags;
        const bool changed = env_step<KJ>(p, iv, s, env, lane, action, raw, reinterpret_cast<int *>(w.scratch));
        s.flags = jss_uniform(s.flags);
        if (SAMPLE) {
            const uint32_t h = jss_hash_env(a.hash_key, p.env_id_base + (uint64_t)env);   // == jss_hash3(seed, genv, step_index)
            const int nxt = env_select_action<KJ, SAMPLE == 1>(iv, s, lane, a.rule, a.coin_mode, h, a.cr_factor);
            if (lane == 0) a.actions_out[env] = nxt;
        }
        if (changed) {
            env_store_to<KJ>(p, iv, w.state_out, lane, s);
            env_emit_all<KJ, true>(p, iv, s, env, lane, w.scratch, raw, w.scratch_sa,
                                   p.state + (size_t)env * blk16 * 4, w.state_out_sa, blk16 * 16u);
        } else if (s.flags != flags_in) {                // only the sticky error bit changed
            if (lane == 0) {
                p.state[(size_t)p.hdr_off16[env] * 4 + JSS_HDR_FLAGS] = (int32_t)s.flags;
                reinterpret_cast<int4 *>(p.scalars)[env] =
                    make_int4(0, 0, s.t, (int)((s.flags << 8) | (s.flags & JSS_FLAG_DONE)));
            }
        }
        buf ^= 1u;
    }
    if (lane == 0) jss_bulk_store_wait_all();            // shared memory must outlive the bulk reads
}

// generator mode: every env's current instance as machine / duration arrays [N][J][M]
__global__ void jss_gen_unpack_kernel(const JssGenParams g, int32_t *machine, int32_t *duration) {
    const size_t jm = (size_t)g.J * g.M, total = (size_t)g.n_envs * jm;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t e = i / jm, q = i % jm;
        const uint32_t op = reinterpret_cast<const uint16_t *>(g.tables + e * g.tbl_bytes + JSS_GEN_HDR_BYTES)[q];
        if (machine) machine[i] = (int32_t)(op >> JSS_OP_SHIFT);
        if (duration) duration[i] = (int32_t)(op & JSS_OP_DMASK);
    }
}

// ---- SM-driven copy of small results into mapped pinned host memory -------------------------
// (mask + scalar records, ~8 MB per step at N = 65 536).  Posted PCIe writes from the SMs do not
// queue behind the 183 MB observation transfer that occupies the D2H copy engine.
__global__ void jss_copy16_kernel(uint4 *dst, const uint4 *src, size_t n16) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x)
        dst[i] = src[i];
}

// ---- per-shard statistics ------------------------------------------------------------------
__global__ void jss_stats_kernel(const JssParams p, unsigned long long *out) {
    // out[0..7] pre-initialised by the host: sums 0, min = ~0ull
    unsigned long long ep = 0, steps = 0, smk = 0, ndone = 0, nerr = 0;
    long long sret = 0;
    unsigned long long mn = ~0ull, mx = 0;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < p.n_envs; e += gridDim.x * blockDim.x) {
        const int64_t *acc = p.acc + (size_t)e * 4;
        const int32_t *hdr = p.state + (size_t)p.hdr_off16[e] * 4;
        ep += (unsigned long long)p.episode_count[e];
        steps += (unsigned long long)acc[0] + (unsigned long long)(((uint32_t)hdr[JSS_HDR_FLAGS] & JSS_FLAG_DONE) ? 0 : hdr[JSS_HDR_EP_STEPS]);
        smk += (unsigned long long)acc[1];
        sret += acc[2];
        if (p.episode_count[e] > 0) {
            const uint64_t mm = (uint64_t)acc[3];
            mn = min(mn, (unsigned long long)(mm >> 32));
            mx = max(mx, (unsigned long long)(mm & 0xffffffffull));
        }
        ndone += ((uint32_t)hdr[JSS_HDR_FLAGS] & JSS_FLAG_DONE) ? 1 : 0;
        nerr += ((uint32_t)hdr[JSS_HDR_FLAGS] & JSS_FLAG_ERROR) ? 1 : 0;
    }
    atomicAdd(&out[0], ep);
    atomicAdd(&out[1], steps);
    atomicAdd(&out[2], smk);
    atomicMin(&out[3], mn);
    atomicMax(&out[4], mx);
    atomicAdd(&out[5], (unsigned long long)sret);
    atomicAdd(&out[6], ndone);
    atomicAdd(&out[7], nerr);
}
