// jss_api.cu -- the C-ABI of include/jss_b200.h on top of the sm_100a kernels in
// jss_device.cuh.  Host side only does: validation, packing of the instance tables,
// grouping envs into per-instance tiles, buffer ownership and kernel launches.
// There is no CPU implementation of the environment in this library.
#ifdef JSS_EMU
#include "cuda_shim.h"  // tests/emu: TEST-ONLY host emulation, never defined for the product build
#else
#include <cuda_runtime.h>
#define JSS_SMEM_DECL(name) extern __shared__ uint4 name[]
#define JSS_LAUNCH(kern, grid, block, smem, stream, ...) kern<<<grid, block, smem, stream>>>(__VA_ARGS__)
// launch with programmatic stream serialization (PDL): the kernel may start its prologue while the preceding
// kernel in the stream drains; it calls griddepcontrol.wait before touching anything mutable
template <typename... KArgs, typename... Args>
static cudaError_t jss_launch_pdl(void (*kern)(KArgs...), int grid, int block, size_t smem, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3((unsigned)block);
    cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}
#define JSS_LAUNCH_PDL(kern, grid, block, smem, stream, ...) jss_launch_pdl(kern, grid, block, smem, stream, __VA_ARGS__)
#endif
#ifdef JSS_EMU
#define JSS_LAUNCH_PDL(kern, grid, block, smem, stream, ...) (JSS_LAUNCH(kern, grid, block, smem, stream, __VA_ARGS__), cudaSuccess)
#endif

#include <algorithm>
#include <climits>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <sched.h>
#include <cctype>
#include <vector>

#include "jss_device.cuh"
#include "jss_host.h"

namespace {

std::string g_create_error;

struct HostInst {
    int J, M;
    int64_t max_time_op, max_time_jobs, sum_op;
    std::vector<int32_t> len;      // jobs_length (host copy: the packed-observation expansion needs it)
};

}  // namespace

struct jss_handle {
    int device = -1;
    int n_envs = 0;
    uint32_t create_flags = 0;
    uint64_t env_id_base = 0;
    int sm_count = 0;
    std::string err;
    int64_t launches = 0;
    double cr_factor = 1.5;                        // CriticalRatio(due_date_factor), dispatching.py:337

    std::vector<HostInst> insts;
    std::vector<JssInstDesc> descs;
    bool loaded = false, assigned = false;

    // device allocations
    std::vector<void *> allocs;
    void *host_block = nullptr;                    // JSS_CREATE_HOST_MIRROR: pinned + mapped block behind the outputs
    int32_t *mirror_actions = nullptr;
    JssInstDesc *d_inst = nullptr;
    uint16_t *d_ops = nullptr, *d_rem = nullptr;
    int32_t *d_len = nullptr;
    unsigned long long *d_stats = nullptr;

    JssParams p{};
    // generator mode (jss_assign_generated): per-env instance tables, regenerated on the device at every reset
    bool gen = false;
    JssGenParams g{};
    int gen_grid[24] = {0};                        // resident-CTA grids of the generator-mode kernel variants (filled lazily)
    JssSmemLayout sl_env{}, sl_step{}, sl_step_rem{};   // shared-memory layouts of the generic / step kernels (step: without / with the suffix-sum table)
    int class_tile_begin[4] = {0, 0, 0, 0}, class_tile_end[4] = {0, 0, 0, 0};  // KJ = 1, 2, 4, 8
    int step_grid[24] = {0};
    int env_grid[16] = {0};                         // resident CTAs per SM of the generic kernel variants (filled lazily)                        // resident-CTA grids of the step kernel variants (filled lazily)
    bool use_pdl = true;
    std::vector<int32_t> env_inst;

    // host-buffer stepping
    int32_t *dev_actions = nullptr;
    float *obs_staging = nullptr;                  // pipelined mode: device copy the D2H engine reads from
    uint8_t *wire[2] = {nullptr, nullptr};         // packed mode: two alternating device rows buffers [N][wire_stride]
    int64_t wire_stride = 0;
    cudaStream_t s_compute = nullptr, s_copy = nullptr;
    cudaEvent_t ev_mask = nullptr, ev_staged = nullptr, ev_wire = nullptr, ev_obs[2] = {nullptr, nullptr};
    int pipe_cur = 0;                              // which ev_obs belongs to the latest begin
    bool pipe_ready = false;
};

namespace {

int fail(jss_t *h, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (h) h->err = buf; else g_create_error = buf;
    return code;
}

#define JSS_CUDA(h, expr)                                                                           \
    do {                                                                                            \
        cudaError_t e_ = (expr);                                                                    \
        if (e_ != cudaSuccess)                                                                      \
            return fail((h), JSS_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_),  \
                        __FILE__, __LINE__);                                                        \
    } while (0)

template <typename T>
int dev_alloc(jss_t *h, T **out, size_t count, bool zero = true) {
    void *ptr = nullptr;
    const size_t bytes = std::max<size_t>(count * sizeof(T), 16);
    JSS_CUDA(h, cudaMalloc(&ptr, bytes));
    h->allocs.push_back(ptr);
    if (zero) JSS_CUDA(h, cudaMemset(ptr, 0, bytes));
    *out = static_cast<T *>(ptr);
    return JSS_OK;
}

inline int round_up(int x, int m) { return (x + m - 1) / m * m; }
inline int kj_of(int J) { return J <= 32 ? 1 : (J <= 64 ? 2 : (J <= 128 ? 4 : 8)); }
inline int class_of(int kj) { return kj == 1 ? 0 : (kj == 2 ? 1 : (kj == 4 ? 2 : 3)); }
// state-block geometry of an instance (must match jss_fill_sminst): per-lane slices are whole vectors
inline int jcap_of(int J) { return J > 128 ? round_up(J, 8) : round_up(J, 4); }
inline int block_words_of(int J, int M) { return 5 * jcap_of(J) + round_up(M, 4) + (J > 128 ? 16 : 8) + 4; }
inline int hdr_word_of(int J, int M) { return 5 * jcap_of(J) + round_up(M, 4) + (J > 128 ? 16 : 8); }

size_t smem_bytes(const JssSmemLayout &sl) { return (size_t)sl.off_warp0 + (size_t)JSS_WARPS_PER_CTA * sl.warp_stride; }

void fill_uni(const JssInstDesc &d, SmInst &u) {
    u.J = d.J; u.M = d.M; u.max_time_op = d.max_time_op; u.max_time_jobs = d.max_time_jobs; u.sum_op = d.sum_op;
    u.f_mto = (float)d.max_time_op; u.f_mtj = (float)d.max_time_jobs; u.f_sop = (float)d.sum_op; u.f_M = (float)d.M;
    u.r_mto = d.r_mto; u.r_mtj = d.r_mtj; u.r_sop = d.r_sop; u.r_M = d.r_M;
    u.Jcap = jcap_of(d.J); u.Mcap = round_up(d.M, 4); u.block_words = block_words_of(d.J, d.M);
    u.n14[0] = u.n14[1] = -u.f_mto; u.r14[0] = u.r14[1] = d.r_mto;
    u.n23[0] = -u.f_M; u.n23[1] = -u.f_mtj; u.r23[0] = d.r_M; u.r23[1] = d.r_mtj;
    u.n56[0] = u.n56[1] = -u.f_sop; u.r56[0] = u.r56[1] = d.r_sop;
}

template <typename Kern>
int step_grid_for(jss_t *h, Kern kern, int slot, size_t smem) {
    int &grid = h->step_grid[slot];
    if (grid == 0) {                                     // once per handle: opt-in smem + occupancy
        if (smem > 48 * 1024)
            JSS_CUDA(h, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int per_sm = 0;
        JSS_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, JSS_WARPS_PER_CTA * 32, smem));
        if (per_sm < 1) return fail(h, JSS_ERR_CUDA, "step kernel does not fit on an SM (smem %zu B)", smem);
        grid = h->sm_count * per_sm;
    }
    return JSS_OK;
}

// uniform batch: one instance, static strided tiles
template <int KJ, int SAMPLE>
int launch_step_uniform(jss_t *h, const JssLaunch &a_in, bool want_rem, cudaStream_t st) {
    JssLaunch a = a_in;
    fill_uni(h->descs[h->p.uniform_inst], a.uni);
    a.tile_begin = 0;
    a.tile_end = (h->n_envs + JSS_WARPS_PER_CTA - 1) / JSS_WARPS_PER_CTA;
    const JssSmemLayout &sl = want_rem ? h->sl_step_rem : h->sl_step;
    const size_t smem = smem_bytes(sl);
    auto kern = jss_step_kernel<KJ, SAMPLE>;
    const int slot = class_of(KJ) * 4 + SAMPLE + (want_rem ? 1 : 0);
    int rc = step_grid_for(h, kern, slot, smem);
    if (rc) return rc;
    const int grid = std::min(a.tile_end, h->step_grid[slot]);
    if (h->use_pdl) JSS_CUDA(h, JSS_LAUNCH_PDL(kern, grid, JSS_WARPS_PER_CTA * 32, smem, st, h->p, a, sl));
    else JSS_LAUNCH(kern, grid, JSS_WARPS_PER_CTA * 32, smem, st, h->p, a, sl);
    JSS_CUDA(h, cudaGetLastError());
    h->launches += 1;
    return JSS_OK;
}

// mixed batch: ONE launch over all lane classes, chunks handed out by ticket
template <int SAMPLE, bool BIG>
int launch_step_mixed(jss_t *h, const JssLaunch &a_in, bool want_rem, cudaStream_t st) {
    JssLaunch a = a_in;
    const JssSmemLayout &sl = want_rem ? h->sl_step_rem : h->sl_step;
    const size_t smem = smem_bytes(sl);
    auto kern = jss_step_mixed_kernel<SAMPLE, BIG>;
    const int slot = (BIG ? 20 : 16) + SAMPLE + (want_rem ? 1 : 0);
    int rc = step_grid_for(h, kern, slot, smem);
    if (rc) return rc;
    const int grid = h->p.n_cta_ranges;                   // one CTA per range (all resident: SMs x 3)
    if (h->use_pdl) JSS_CUDA(h, JSS_LAUNCH_PDL(kern, grid, JSS_WARPS_PER_CTA * 32, smem, st, h->p, a, sl));
    else JSS_LAUNCH(kern, grid, JSS_WARPS_PER_CTA * 32, smem, st, h->p, a, sl);
    JSS_CUDA(h, cudaGetLastError());
    h->launches += 1;
    return JSS_OK;
}

int launch_step(jss_t *h, const JssLaunch &a, cudaStream_t st) {
    const bool rem = a.rule == JSS_RULE_MWR || a.rule == JSS_RULE_LWR || a.rule == JSS_RULE_CR;
    const int sample = a.actions_out == nullptr ? 0 : (a.rule == JSS_RULE_RANDOM ? 1 : 2);
    if (h->p.uniform_inst < 0) {
        const bool big = h->class_tile_end[3] > h->class_tile_begin[3];     // instances with 129..256 jobs in the batch
        if (big) {
            if (sample == 0) return launch_step_mixed<0, true>(h, a, false, st);
            if (sample == 1) return launch_step_mixed<1, true>(h, a, false, st);
            return launch_step_mixed<2, true>(h, a, rem, st);
        }
        if (sample == 0) return launch_step_mixed<0, false>(h, a, false, st);
        if (sample == 1) return launch_step_mixed<1, false>(h, a, false, st);
        return launch_step_mixed<2, false>(h, a, rem, st);
    }
    const int kj = kj_of(h->insts[h->p.uniform_inst].J);
#define JSS_STEP_UNI(KJ_)                                                               \
    do {                                                                                \
        if (sample == 0) return launch_step_uniform<KJ_, 0>(h, a, false, st);           \
        if (sample == 1) return launch_step_uniform<KJ_, 1>(h, a, false, st);           \
        return launch_step_uniform<KJ_, 2>(h, a, rem, st);                              \
    } while (0)
    if (kj == 1) JSS_STEP_UNI(1);
    if (kj == 2) JSS_STEP_UNI(2);
    if (kj == 4) JSS_STEP_UNI(4);
    JSS_STEP_UNI(8);
#undef JSS_STEP_UNI
}

template <int KJ, int MODE>
int launch_variant(jss_t *h, const JssLaunch &a, const JssSmemLayout &sl, cudaStream_t st) {
    const int n_tiles = a.tile_end - a.tile_begin;
    const size_t smem = smem_bytes(sl);
    auto kern = jss_env_kernel<KJ, MODE>;
    // once per handle and kernel variant: opt-in to > 48 KB of dynamic shared memory, resident CTAs per SM
    int &per_sm = h->env_grid[class_of(KJ) * 4 + (MODE == JSS_MODE_RESET ? 0 : MODE == JSS_MODE_ROLLOUT ? 1 : 2)];
    if (per_sm == 0) {
        if (smem > 48 * 1024)
            JSS_CUDA(h, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        JSS_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, JSS_WARPS_PER_CTA * 32, smem));
        if (per_sm < 1) { per_sm = 0; return fail(h, JSS_ERR_CUDA, "kernel does not fit on an SM (smem %zu B)", smem); }
    }
    // policy kernels touch ~50 B per env: latency-bound, so give every tile its own CTA
    // instead of a persistent loop with a dependent load per iteration
    const int grid = (MODE == JSS_MODE_POLICY) ? n_tiles : std::min(n_tiles, h->sm_count * per_sm);
    JSS_LAUNCH(kern, grid, JSS_WARPS_PER_CTA * 32, smem, st, h->p, a, sl);
    JSS_CUDA(h, cudaGetLastError());
    h->launches += 1;
    return JSS_OK;
}

template <int KJ>
int launch_class(jss_t *h, const JssLaunch &a, const JssSmemLayout &sl, cudaStream_t st) {
    if (a.tile_end - a.tile_begin <= 0) return JSS_OK;
    switch (a.mode) {
    case JSS_MODE_POLICY: return launch_variant<KJ, JSS_MODE_POLICY>(h, a, sl, st);
    case JSS_MODE_ROLLOUT: return launch_variant<KJ, JSS_MODE_ROLLOUT>(h, a, sl, st);
    default: return launch_variant<KJ, JSS_MODE_RESET>(h, a, sl, st);   // reset / export / import
    }
}

// ---- generator mode -------------------------------------------------------------------------------
template <typename Kern>
int gen_grid_for(jss_t *h, Kern kern, int slot, int threads, size_t smem) {
    int &grid = h->gen_grid[slot];
    if (grid == 0) {
        if (smem > 48 * 1024)
            JSS_CUDA(h, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int per_sm = 0;
        JSS_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem));
        if (per_sm < 1) return fail(h, JSS_ERR_CUDA, "generator-mode kernel does not fit on an SM (smem %zu B)", smem);
        grid = h->sm_count * per_sm;
    }
    return JSS_OK;
}

template <int KJ, int SAMPLE>
int launch_gen_step(jss_t *h, const JssLaunch &a_in, cudaStream_t st) {
    JssLaunch a = a_in;
    fill_uni(h->descs[0], a.uni);                        // the batch geometry (every env has the same shape)
    JssGenStepArgs ga;
    ga.sl = h->sl_step;                                  // no CTA-shared tables: the warp regions start at 0
    ga.sl.off_warp0 = 0;
    ga.g = h->g;
    ga.g.off_gen = ga.sl.warp_stride;
    ga.sl.warp_stride += (int32_t)sizeof(SmInst) + 2 * ga.g.tbl_bytes;
    const size_t smem = (size_t)JSS_GEN_STEP_WARPS * ga.sl.warp_stride;
    auto kern = jss_gen_step_kernel<KJ, SAMPLE>;
    int rc = gen_grid_for(h, kern, class_of(KJ) * 4 + SAMPLE, JSS_GEN_STEP_WARPS * 32, smem);
    if (rc) return rc;
    const int grid = std::min(h->gen_grid[class_of(KJ) * 4 + SAMPLE], (h->n_envs + JSS_GEN_STEP_WARPS - 1) / JSS_GEN_STEP_WARPS);
    if (h->use_pdl) JSS_CUDA(h, JSS_LAUNCH_PDL(kern, grid, JSS_GEN_STEP_WARPS * 32, smem, st, h->p, a, ga));
    else JSS_LAUNCH(kern, grid, JSS_GEN_STEP_WARPS * 32, smem, st, h->p, a, ga);
    JSS_CUDA(h, cudaGetLastError());
    h->launches += 1;
    return JSS_OK;
}

template <int KJ, int MODE>
int launch_gen_env(jss_t *h, const JssLaunch &a_in, cudaStream_t st) {
    JssLaunch a = a_in;
    a.tile_begin = 0;
    a.tile_end = (h->n_envs + JSS_WARPS_PER_CTA - 1) / JSS_WARPS_PER_CTA;
    JssGenParams g = h->g;
    g.warp_stride = (int32_t)sizeof(SmInst) + h->sl_env.scratch_words * 4;
    const size_t smem = (size_t)JSS_WARPS_PER_CTA * g.warp_stride;
    auto kern = jss_gen_env_kernel<KJ, MODE>;
    const int slot = 12 + class_of(KJ) * 4 + (MODE == JSS_MODE_RESET ? 0 : MODE == JSS_MODE_ROLLOUT ? 1 : 2);
    int rc = gen_grid_for(h, kern, slot, JSS_WARPS_PER_CTA * 32, smem);
    if (rc) return rc;
    // policy launches: latency-bound, one CTA per tile (as launch_variant)
    const int grid = (MODE == JSS_MODE_POLICY) ? a.tile_end : std::min(a.tile_end, h->gen_grid[slot]);
    JSS_LAUNCH(kern, grid, JSS_WARPS_PER_CTA * 32, smem, st, h->p, a, g);
    JSS_CUDA(h, cudaGetLastError());
    h->launches += 1;
    return JSS_OK;
}

template <int KJ>
int launch_gen_class(jss_t *h, const JssLaunch &a, cudaStream_t st) {
    if (a.mode == JSS_MODE_STEP) {
        const int sample = a.actions_out == nullptr ? 0 : (a.rule == JSS_RULE_RANDOM ? 1 : 2);
        if (sample == 0) return launch_gen_step<KJ, 0>(h, a, st);
        if (sample == 1) return launch_gen_step<KJ, 1>(h, a, st);
        return launch_gen_step<KJ, 2>(h, a, st);
    }
    if (a.mode == JSS_MODE_POLICY) return launch_gen_env<KJ, JSS_MODE_POLICY>(h, a, st);
    if (a.mode == JSS_MODE_ROLLOUT) return launch_gen_env<KJ, JSS_MODE_ROLLOUT>(h, a, st);
    return launch_gen_env<KJ, JSS_MODE_RESET>(h, a, st);   // reset / export
}

int launch_gen(jss_t *h, const JssLaunch &a, cudaStream_t st) {
    const int kj = kj_of(h->g.J);
    if (kj == 1) return launch_gen_class<1>(h, a, st);
    if (kj == 2) return launch_gen_class<2>(h, a, st);
    return launch_gen_class<4>(h, a, st);
}

int launch_all(jss_t *h, JssLaunch a, bool want_rem, cudaStream_t st) {
    if (h->gen) return launch_gen(h, a, st);
    if (a.mode == JSS_MODE_STEP && !a.export_after) return launch_step(h, a, st);   // one launch, whatever the mix of lane classes
    (void)want_rem;
    const JssSmemLayout &sl = h->sl_env;
    for (int c = 0; c < 4; c++) {
        a.tile_begin = h->class_tile_begin[c];
        a.tile_end = h->class_tile_end[c];
        int rc = JSS_OK;
        if (c == 0) rc = launch_class<1>(h, a, sl, st);
        else if (c == 1) rc = launch_class<2>(h, a, sl, st);
        else if (c == 2) rc = launch_class<4>(h, a, sl, st);
        else rc = launch_class<8>(h, a, sl, st);
        if (rc != JSS_OK) return rc;
    }
    return JSS_OK;
}

bool rule_wants_rem(int rule) { return rule == JSS_RULE_MWR || rule == JSS_RULE_LWR || rule == JSS_RULE_CR; }

int check_ready(jss_t *h) {
    if (!h) return JSS_ERR_INVALID;
    if (!h->assigned) return fail(h, JSS_ERR_STATE, "jss_load_instances + jss_assign must be called first");
    JSS_CUDA(h, cudaSetDevice(h->device));
    return JSS_OK;
}

}  // namespace

extern "C" {

int jss_abi_version(void) { return JSS_ABI_VERSION; }

const char *jss_last_error(const jss_t *h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int64_t jss_launch_count(const jss_t *h) { return h ? h->launches : 0; }

int jss_set_cr_due_date_factor(jss_t *h, double factor) {
    if (!h || !(factor == factor)) return fail(h, JSS_ERR_INVALID, "jss_set_cr_due_date_factor: bad arguments");
    h->cr_factor = factor;
    return JSS_OK;
}

int jss_create(jss_t **out, int device, int n_envs, uint32_t flags, uint64_t env_id_base) {
    if (!out || n_envs <= 0) return fail(nullptr, JSS_ERR_INVALID, "jss_create: bad arguments");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, JSS_ERR_NO_DEVICE,
                    "no CUDA device (%s); this library has no CPU fallback", cudaGetErrorString(e));
    if (device < 0 || device >= ndev)
        return fail(nullptr, JSS_ERR_NO_DEVICE, "device %d out of range (have %d)", device, ndev);
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess)
        return fail(nullptr, JSS_ERR_NO_DEVICE, "cudaGetDeviceProperties failed");
    if (prop.major < 10)
        return fail(nullptr, JSS_ERR_NO_DEVICE, "device %d is sm_%d%d; this build targets sm_100a (B200)", device,
                    prop.major, prop.minor);
    jss_t *h = new jss_handle();
    h->device = device;
    h->n_envs = n_envs;
    h->create_flags = flags;
    h->env_id_base = env_id_base;
    h->sm_count = prop.multiProcessorCount;
    if (cudaSetDevice(device) != cudaSuccess) {
        delete h;
        return fail(nullptr, JSS_ERR_CUDA, "cudaSetDevice(%d) failed", device);
    }
    *out = h;
    return JSS_OK;
}

void jss_destroy(jss_t *h) {
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->pipe_ready) {
        cudaStreamSynchronize(h->s_compute); cudaStreamSynchronize(h->s_copy);
        cudaEventDestroy(h->ev_mask); cudaEventDestroy(h->ev_staged); cudaEventDestroy(h->ev_wire); cudaEventDestroy(h->ev_obs[0]); cudaEventDestroy(h->ev_obs[1]);
        cudaStreamDestroy(h->s_compute); cudaStreamDestroy(h->s_copy);
    }
    for (void *ptr : h->allocs) cudaFree(ptr);
    if (h->host_block) cudaFreeHost(h->host_block);
    delete h;
}

int jss_load_instances(jss_t *h, int n_inst, const int32_t *jobs, const int32_t *machines, const int64_t *offsets,
                       const int32_t *machine, const int32_t *duration) {
    if (!h || n_inst <= 0 || !jobs || !machines || !offsets || !machine || !duration)
        return fail(h, JSS_ERR_INVALID, "jss_load_instances: bad arguments");
    if (h->loaded) return fail(h, JSS_ERR_STATE, "instances already loaded");
    if (n_inst >= (1 << 23)) return fail(h, JSS_ERR_UNSUPPORTED, "too many instances");
    JSS_CUDA(h, cudaSetDevice(h->device));
    std::vector<uint16_t> ops, rem;
    std::vector<int32_t> len;
    h->insts.resize(n_inst);
    h->descs.resize(n_inst);
    for (int k = 0; k < n_inst; k++) {
        const int J = jobs[k], M = machines[k];
        if (J <= 0 || M <= 1)  // asserts at jss_env.py:93-94
            return fail(h, JSS_ERR_INVALID, "instance %d: need jobs > 0 and machines > 1 (got %dx%d)", k, J, M);
        if (J > JSS_MAX_JOBS || M > JSS_MAX_MACHINES)
            return fail(h, JSS_ERR_UNSUPPORTED, "instance %d: %dx%d exceeds the %dx%d kernel limit", k, J, M,
                        JSS_MAX_JOBS, JSS_MAX_MACHINES);
        const int32_t *mm = machine + offsets[k], *dd = duration + offsets[k];
        HostInst hi{J, M, 0, 0, 0, std::vector<int32_t>((size_t)J)};
        JssInstDesc d{};
        d.J = J; d.M = M;
        d.ops_off = (int32_t)ops.size();
        d.len_off = (int32_t)len.size();
        d.rem_off = (int32_t)rem.size();
        ops.resize(ops.size() + round_up(J * M, 8), 0);
        len.resize(len.size() + round_up(J, 4), 0);
        rem.resize(rem.size() + round_up(J * (M + 1), 8), 0);
        for (int q = 0; q < J * M; q++) {
            const int m = mm[q], t = dd[q];
            if (m < 0 || m >= M) return fail(h, JSS_ERR_INVALID, "instance %d: machine %d out of range", k, m);
            // Zero-length ops are rejected: the reference itself cannot finish such an episode -- an allocated op of
            // duration 0 never satisfies `was_left_time > 0` (jss_env.py:529), so the job never advances to its
            // next op and is re-legalised on the same machine at the same instant (jss_env.py:616-634).
            if (t < 1 || t > JSS_MAX_DURATION)
                return fail(h, JSS_ERR_UNSUPPORTED, "instance %d: duration %d outside [1, %d]", k, t, JSS_MAX_DURATION);
        }
        for (int j = 0; j < J; j++) {
            // tables + scalars of the row: the same code the device generator runs (jss_gen.h)
            int32_t mx = 0;
            const int32_t total = jss_pack_job_row(mm + j * M, dd + j * M, M, &ops[d.ops_off + j * M],
                                                   &rem[d.rem_off + j * (M + 1)], &mx);
            len[d.len_off + j] = total;                                 // jss_env.py:87
            hi.len[j] = total;
            hi.max_time_op = std::max<int64_t>(hi.max_time_op, mx);    // jss_env.py:86
            hi.sum_op += total;                                         // jss_env.py:88
            hi.max_time_jobs = std::max<int64_t>(hi.max_time_jobs, total);   // jss_env.py:89
        }
        const int32_t ops_off = d.ops_off, len_off = d.len_off, rem_off = d.rem_off;
        d = jss_inst_desc(J, M, (int32_t)hi.max_time_op, (int32_t)hi.max_time_jobs, (int32_t)hi.sum_op);
        d.ops_off = ops_off; d.len_off = len_off; d.rem_off = rem_off;
        h->insts[k] = hi;
        h->descs[k] = d;
    }
    int rc;
    if ((rc = dev_alloc(h, &h->d_inst, (size_t)n_inst))) return rc;
    if ((rc = dev_alloc(h, &h->d_ops, ops.size()))) return rc;
    if ((rc = dev_alloc(h, &h->d_len, len.size()))) return rc;
    if ((rc = dev_alloc(h, &h->d_rem, rem.size()))) return rc;
    JSS_CUDA(h, cudaMemcpy(h->d_inst, h->descs.data(), sizeof(JssInstDesc) * n_inst, cudaMemcpyHostToDevice));
    JSS_CUDA(h, cudaMemcpy(h->d_ops, ops.data(), ops.size() * 2, cudaMemcpyHostToDevice));
    JSS_CUDA(h, cudaMemcpy(h->d_len, len.data(), len.size() * 4, cudaMemcpyHostToDevice));
    JSS_CUDA(h, cudaMemcpy(h->d_rem, rem.data(), rem.size() * 2, cudaMemcpyHostToDevice));
    h->loaded = true;
    return JSS_OK;
}

int jss_instance_scalars(jss_t *h, int inst, int64_t out[3]) {
    if (h && h->gen)
        return fail(h, JSS_ERR_UNSUPPORTED, "jss_instance_scalars: generator mode has no instance list (see jss_get_env_instances)");
    if (!h || !out || !h->loaded || inst < 0 || inst >= (int)h->insts.size())
        return fail(h, JSS_ERR_INVALID, "jss_instance_scalars: bad arguments");
    out[0] = h->insts[inst].max_time_op;
    out[1] = h->insts[inst].max_time_jobs;
    out[2] = h->insts[inst].sum_op;
    return JSS_OK;
}

}  // extern "C"

namespace {
// grouping, shared-memory layouts and every per-env buffer of a batch whose instances are loaded (jss_assign), or
// whose shape is (jss_assign_generated); ends with the first reset
int assign_impl(jss_t *h, const int32_t *env_to_inst) {
    JSS_CUDA(h, cudaSetDevice(h->device));
    const int N = h->n_envs, n_inst = (int)h->insts.size();
    int jmax = 0, mmax = 0, ops_max = 0, rem_max = 0;
    h->env_inst.assign(env_to_inst, env_to_inst + N);
    std::vector<char> used(n_inst, 0);
    for (int e = 0; e < N; e++) {
        const int k = env_to_inst[e];
        if (k < 0 || k >= n_inst) return fail(h, JSS_ERR_INVALID, "env %d: instance %d out of range", e, k);
        used[k] = 1;
    }
    for (int k = 0; k < n_inst; k++) {
        if (!used[k]) continue;
        jmax = std::max(jmax, h->insts[k].J);
        mmax = std::max(mmax, h->insts[k].M);
        ops_max = std::max(ops_max, h->insts[k].J * h->insts[k].M);
        rem_max = std::max(rem_max, h->insts[k].J * (h->insts[k].M + 1));
    }
    // group envs by (KJ class, instance) -> tiles of <= JSS_WARPS_PER_CTA envs of one instance.  The most
    // expensive lane class (KJ = 4) comes first: the mixed-batch step kernel hands the tile list out front to
    // back, so the cheap 15..30-job envs fill the tail (longest processing time first).
    std::vector<int32_t> order(N);
    for (int e = 0; e < N; e++) order[e] = e;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) {
        const int ka = env_to_inst[a], kb = env_to_inst[b];
        const int ca = class_of(kj_of(h->insts[ka].J)), cb = class_of(kj_of(h->insts[kb].J));
        if (ca != cb) return ca > cb;
        return ka < kb;
    });
    std::vector<JssTile> tiles;
    std::vector<uint32_t> state_off16((size_t)N), hdr_off16((size_t)N);
    std::vector<double> tile_cost;
    for (int c = 0; c < 4; c++) h->class_tile_begin[c] = h->class_tile_end[c] = 0;
    int pos = 0;
    int cur_class = -1;
    uint64_t off16 = 0;                                  // running state offset in 16-byte units
    while (pos < N) {
        const int k = env_to_inst[order[pos]];
        const int c = class_of(kj_of(h->insts[k].J));
        const uint32_t block16 = (uint32_t)block_words_of(h->insts[k].J, h->insts[k].M) / 4;
        const uint32_t hdr16 = (uint32_t)hdr_word_of(h->insts[k].J, h->insts[k].M) / 4;
        int end = pos;
        while (end < N && env_to_inst[order[end]] == k) end++;
        if (c != cur_class) {
            if (cur_class >= 0) h->class_tile_end[cur_class] = (int)tiles.size();
            h->class_tile_begin[c] = (int)tiles.size();
            cur_class = c;
        }
        for (int f = pos; f < end; f += JSS_WARPS_PER_CTA) {
            JssTile t;
            const int cnt = std::min(JSS_WARPS_PER_CTA, end - f);
            t.first = f;
            t.inst_count = (k << 8) | cnt;
            t.state_off16 = (uint32_t)off16;
            t.block16 = block16;
            for (int w = 0; w < cnt; w++) {
                state_off16[order[f + w]] = (uint32_t)(off16 + (uint64_t)w * block16);
                hdr_off16[order[f + w]] = (uint32_t)(off16 + (uint64_t)w * block16) + hdr16;
            }
            off16 += (uint64_t)cnt * block16;
            tiles.push_back(t);
            // relative cost of an env-step: measured on uniform batches it is ~linear in J (issue-bound kernel)
            tile_cost.push_back(cnt * (40.0 + h->insts[k].J));
        }
        pos = end;
    }
    if (cur_class >= 0) h->class_tile_end[cur_class] = (int)tiles.size();
    if (off16 >= (1ull << 32)) return fail(h, JSS_ERR_UNSUPPORTED, "state exceeds 64 GiB");
    const size_t state_words = (size_t)off16 * 4;

    // mixed-batch step kernel: every persistent CTA gets an equal slice of EVERY lane class (tile counts differ by at
    // most one per class; the extras are dithered with a different phase per class so that no CTA collects them all)
    std::vector<JssCtaRange> ranges;
    {
        const int n_cta = std::max(1, std::min((int)tiles.size(), h->sm_count * JSS_MIN_CTAS));
        ranges.resize((size_t)n_cta);
        for (int c = 0; c < 4; c++) {                     // c = 3: KJ = 8, c = 2: KJ = 4, c = 1: KJ = 2, c = 0: KJ = 1
            const int tb = h->class_tile_begin[c], n = h->class_tile_end[c] - tb;
            const int shift = (c * n_cta) / 4;            // CTA that starts this class's Bresenham sequence
            int given = 0;
            for (int k = 0; k < n_cta; k++) {
                const int b = (k + shift) % n_cta;
                const int upto = (int)(((int64_t)(k + 1) * n) / n_cta);
                int32_t *lo = c == 3 ? &ranges[b].a8 : (c == 2 ? &ranges[b].a4 : (c == 1 ? &ranges[b].a2 : &ranges[b].a1));
                lo[0] = tb + given; lo[1] = tb + upto;
                given = upto;
            }
        }
    }

    JssParams &p = h->p;
    p.n_envs = N;
    p.jobs_max = jmax;
    p.machines_max = mmax;
    p.Jcap = jcap_of(jmax);
    p.Mcap = round_up(mmax, 4);
    p.block_words = block_words_of(jmax, mmax);          // batch maximum: sizes the shared-memory staging buffers
    p.mask_stride = round_up(jmax + 1, jmax > 128 ? 8 : 4);   // the 8-jobs-per-lane class stores 8 mask bytes per lane
    p.create_flags = (int32_t)h->create_flags;
    p.env_id_base = h->env_id_base;
    {
        bool uniform = true;
        for (int e = 0; e < N; e++) uniform = uniform && env_to_inst[e] == env_to_inst[0];
        p.uniform_inst = uniform ? env_to_inst[0] : -1;   // then `order` is the identity (stable sort)
    }
    p.inst = h->d_inst; p.ops_pool = h->d_ops; p.len_pool = h->d_len; p.rem_pool = h->d_rem;

    {   // shared-memory layouts: [SmInst][ops u16][len i32][rem u16][per-warp regions], 16-byte aligned regions
        JssSmemLayout sl{};
        sl.off_len = (int32_t)sizeof(SmInst) + round_up(ops_max, 8) * 2;
        sl.off_rem = sl.off_len + round_up(jmax, 4) * 4;
        sl.off_warp0 = sl.off_rem + round_up(rem_max, 8) * 2;
        // observation staging (7 floats per job slot); env_check_no_op (general instances) also keeps its 32-int
        // per-warp machine-horizon table here, so never less than 32 words (tiny instances: 7 * Jcap < 32)
        sl.scratch_words = std::max(7 * p.Jcap, 32);
        h->sl_env = sl;
        h->sl_env.warp_stride = sl.scratch_words * 4;
        h->sl_env.off_scratch = 0;
        h->sl_step_rem = sl;
        h->sl_step_rem.off_scratch = 16 + p.block_words * 4;                               // [mbarrier][state-in]
        h->sl_step_rem.warp_stride = h->sl_step_rem.off_scratch + sl.scratch_words * 4 + p.block_words * 4;   // [scratch][state-out]
        h->sl_step = h->sl_step_rem;                      // launches that stage no suffix sums leave their room to the L1
        h->sl_step.off_warp0 = h->sl_step.off_rem;
    }

    int rc;
    int32_t *d_order = nullptr;
    JssTile *d_tiles = nullptr;
    JssCtaRange *d_ranges = nullptr;
    uint32_t *d_soff = nullptr, *d_hoff = nullptr;
    if ((rc = dev_alloc(h, &d_order, (size_t)N))) return rc;
    if ((rc = dev_alloc(h, &d_tiles, tiles.size()))) return rc;
    if ((rc = dev_alloc(h, &d_ranges, ranges.size()))) return rc;
    if ((rc = dev_alloc(h, &d_soff, (size_t)N))) return rc;
    if ((rc = dev_alloc(h, &d_hoff, (size_t)N))) return rc;
    JSS_CUDA(h, cudaMemcpy(d_order, order.data(), (size_t)N * 4, cudaMemcpyHostToDevice));
    JSS_CUDA(h, cudaMemcpy(d_tiles, tiles.data(), tiles.size() * sizeof(JssTile), cudaMemcpyHostToDevice));
    JSS_CUDA(h, cudaMemcpy(d_ranges, ranges.data(), ranges.size() * sizeof(JssCtaRange), cudaMemcpyHostToDevice));
    JSS_CUDA(h, cudaMemcpy(d_soff, state_off16.data(), (size_t)N * 4, cudaMemcpyHostToDevice));
    JSS_CUDA(h, cudaMemcpy(d_hoff, hdr_off16.data(), (size_t)N * 4, cudaMemcpyHostToDevice));
    p.order = d_order;
    p.tiles = d_tiles;
    p.cta_ranges = d_ranges;
    p.n_cta_ranges = (int32_t)ranges.size();
    p.state_off16 = d_soff;
    p.hdr_off16 = d_hoff;
    const size_t NJ = (size_t)N * jmax, NM = (size_t)N * mmax;
    if ((rc = dev_alloc(h, &p.state, state_words))) return rc;
    if (h->create_flags & JSS_CREATE_HOST_MIRROR) {
        // every per-transition output in one pinned, device-mapped host block (unified addressing: the device
        // pointer equals the host pointer); meant for small batches -- the kernels write over PCIe
        size_t off = 0;
        auto take = [&](size_t bytes) { const size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
        const size_t o_mask = take(N * (size_t)p.mask_stride), o_obs = take(NJ * 7 * 4), o_sc = take((size_t)N * 16);
        const size_t o_i[5] = {take(NJ * 4), take(NJ * 4), take(NJ * 4), take(NJ * 4), take(NJ * 4)};
        const size_t o_tuam = take(NM * 4), o_legal = take(NJ), o_blocked = take(NJ), o_act = take((size_t)N * 4);
        JSS_CUDA(h, cudaHostAlloc(&h->host_block, off, cudaHostAllocMapped | cudaHostAllocPortable));
        memset(h->host_block, 0, off);
        void *dev = nullptr;
        JSS_CUDA(h, cudaHostGetDevicePointer(&dev, h->host_block, 0));
        if (dev != h->host_block) return fail(h, JSS_ERR_CUDA, "host mirror needs unified addressing");
        char *b = static_cast<char *>(h->host_block);
        p.mask = reinterpret_cast<uint8_t *>(b + o_mask); p.obs = reinterpret_cast<float *>(b + o_obs);
        p.scalars = reinterpret_cast<int32_t *>(b + o_sc);
        p.x_todo = reinterpret_cast<int32_t *>(b + o_i[0]); p.x_tufco = reinterpret_cast<int32_t *>(b + o_i[1]);
        p.x_idle_last = reinterpret_cast<int32_t *>(b + o_i[2]); p.x_total_idle = reinterpret_cast<int32_t *>(b + o_i[3]);
        p.x_col4 = reinterpret_cast<int32_t *>(b + o_i[4]); p.x_tuam = reinterpret_cast<int32_t *>(b + o_tuam);
        p.x_legal = reinterpret_cast<uint8_t *>(b + o_legal); p.x_blocked = reinterpret_cast<uint8_t *>(b + o_blocked);
        h->mirror_actions = reinterpret_cast<int32_t *>(b + o_act);
    } else {
        if ((rc = dev_alloc(h, &p.mask, (size_t)N * p.mask_stride))) return rc;
        if ((rc = dev_alloc(h, &p.obs, NJ * 7))) return rc;
        if ((rc = dev_alloc(h, &p.scalars, (size_t)N * 4))) return rc;
        if ((rc = dev_alloc(h, &p.x_todo, NJ))) return rc;
        if ((rc = dev_alloc(h, &p.x_tufco, NJ))) return rc;
        if ((rc = dev_alloc(h, &p.x_idle_last, NJ))) return rc;
        if ((rc = dev_alloc(h, &p.x_total_idle, NJ))) return rc;
        if ((rc = dev_alloc(h, &p.x_col4, NJ))) return rc;
        if ((rc = dev_alloc(h, &p.x_tuam, NM))) return rc;
        if ((rc = dev_alloc(h, &p.x_legal, NJ))) return rc;
        if ((rc = dev_alloc(h, &p.x_blocked, NJ))) return rc;
    }
    if (h->create_flags & JSS_CREATE_RECORD_SOLUTION) {
        if ((rc = dev_alloc(h, &p.solution, NJ * mmax, false))) return rc;
        JSS_CUDA(h, cudaMemset(p.solution, 0xff, NJ * mmax * 4));  // -1
    } else {
        p.solution = nullptr;
    }
    if ((rc = dev_alloc(h, &p.episode_count, (size_t)N))) return rc;
    if ((rc = dev_alloc(h, &p.last_makespan, (size_t)N))) return rc;
    if ((rc = dev_alloc(h, &p.last_return, (size_t)N))) return rc;
    if ((rc = dev_alloc(h, &p.acc, (size_t)N * 4))) return rc;
    if ((rc = dev_alloc(h, &h->d_stats, (size_t)JSS_STATS_LEN))) return rc;
    if ((rc = dev_alloc(h, &h->dev_actions, (size_t)N))) return rc;
    h->assigned = true;
    // a fresh batch starts reset, like a freshly constructed + reset reference env
    return jss_reset(h, nullptr, nullptr);
}
}  // namespace

extern "C" {

int jss_assign(jss_t *h, const int32_t *env_to_inst) {
    if (!h || !env_to_inst) return fail(h, JSS_ERR_INVALID, "jss_assign: bad arguments");
    if (!h->loaded) return fail(h, JSS_ERR_STATE, "jss_load_instances must be called first");
    if (h->assigned) return fail(h, JSS_ERR_STATE, "envs already assigned");
    return assign_impl(h, env_to_inst);
}

namespace {
int check_gen_shape(jss_t *h, int jobs, int machines, int dur_min, int dur_max, const char *what) {
    if (jobs < 1 || machines < 2 || dur_min > dur_max)
        return fail(h, JSS_ERR_INVALID, "%s: need jobs >= 1, machines >= 2 and dur_min <= dur_max (got %dx%d, [%d, %d])",
                    what, jobs, machines, dur_min, dur_max);
    if (jobs > JSS_GEN_MAX_JOBS || machines > JSS_MAX_MACHINES || dur_min < 1 || dur_max > JSS_MAX_DURATION)
        return fail(h, JSS_ERR_UNSUPPORTED, "%s: %dx%d with durations [%d, %d] exceeds the generator limits (%dx%d, [1, %d])",
                    what, jobs, machines, dur_min, dur_max, JSS_GEN_MAX_JOBS, JSS_MAX_MACHINES, JSS_MAX_DURATION);
    return JSS_OK;
}
}  // namespace

int jss_assign_generated(jss_t *h, int jobs, int machines, int dur_min, int dur_max, uint64_t inst_seed) {
    if (!h) return JSS_ERR_INVALID;
    if (h->loaded || h->assigned)
        return fail(h, JSS_ERR_STATE, "jss_assign_generated: takes the place of jss_load_instances + jss_assign on a fresh handle");
    int rc = check_gen_shape(h, jobs, machines, dur_min, dur_max, "jss_assign_generated");
    if (rc) return rc;
    if (h->create_flags & JSS_CREATE_HOST_MIRROR)
        return fail(h, JSS_ERR_UNSUPPORTED, "jss_assign_generated: JSS_CREATE_HOST_MIRROR is not available in generator mode");
    JSS_CUDA(h, cudaSetDevice(h->device));
    // the shape as the one "instance" of a uniform batch: state geometry, identity order and buffers come from it
    const int J = jobs, M = machines, N = h->n_envs;
    h->insts.assign(1, HostInst{J, M, 0, 0, 0, std::vector<int32_t>((size_t)J)});
    JssInstDesc d{};
    d.J = J; d.M = M;
    h->descs.assign(1, d);
    JssGenParams &g = h->g;
    g.J = J; g.M = M; g.dmin = dur_min; g.dmax = dur_max; g.seed = inst_seed;
    g.ops_bytes = 2 * round_up(J * M, 8);
    g.tbl_bytes = JSS_GEN_HDR_BYTES + g.ops_bytes + 4 * round_up(J, 4);
    g.rem_elems = round_up(J * (M + 1), 8);
    g.n_envs = N;
    if ((rc = dev_alloc(h, &g.tables, (size_t)N * g.tbl_bytes))) return rc;
    if ((rc = dev_alloc(h, &g.rem, (size_t)N * g.rem_elems))) return rc;
    if ((rc = dev_alloc(h, &g.index, (size_t)N, false))) return rc;
    JSS_CUDA(h, cudaMemset(g.index, 0xff, (size_t)N * 4));   // -1: the first reset draws instance 0
    h->gen = true;
    h->loaded = true;
    std::vector<int32_t> e2i((size_t)N, 0);
    return assign_impl(h, e2i.data());
}

int jss_get_env_instances(jss_t *h, int32_t *machine_dev, int32_t *duration_dev, int32_t *index_dev, void *stream) {
    int rc = check_ready(h);
    if (rc) return rc;
    if (!h->gen) return fail(h, JSS_ERR_STATE, "jss_get_env_instances: the handle is not in generator mode");
    cudaStream_t st = (cudaStream_t)stream;
    if (machine_dev || duration_dev) {
        const size_t total = (size_t)h->n_envs * h->g.J * h->g.M;
        const int blocks = (int)std::min<size_t>((total + 255) / 256, (size_t)h->sm_count * 8);
        JSS_LAUNCH(jss_gen_unpack_kernel, blocks, 256, 0, st, h->g, machine_dev, duration_dev);
        JSS_CUDA(h, cudaGetLastError());
        h->launches += 1;
    }
    if (index_dev)
        JSS_CUDA(h, cudaMemcpyAsync(index_dev, h->g.index, (size_t)h->n_envs * 4, cudaMemcpyDeviceToDevice, st));
    return JSS_OK;
}

int jss_generate_instance(int jobs, int machines, int dur_min, int dur_max, uint64_t inst_seed, uint64_t env_id,
                          uint64_t index, int32_t *machine_host, int32_t *duration_host) {
    if (!machine_host || !duration_host) return JSS_ERR_INVALID;
    int rc = check_gen_shape(nullptr, jobs, machines, dur_min, dur_max, "jss_generate_instance");
    if (rc) return rc;
    uint8_t mach[JSS_MAX_MACHINES];
    int32_t dur[JSS_MAX_MACHINES];
    for (int j = 0; j < jobs; j++) {
        jss_gen_row(inst_seed, env_id, index, j, machines, dur_min, dur_max, mach, dur);
        for (int i = 0; i < machines; i++) {
            machine_host[j * machines + i] = mach[i];
            duration_host[j * machines + i] = dur[i];
        }
    }
    return JSS_OK;
}

int jss_get_buffers(jss_t *h, jss_buffers *out) {
    if (!h || !out) return JSS_ERR_INVALID;
    if (!h->assigned) return fail(h, JSS_ERR_STATE, "jss_assign must be called first");
    const JssParams &p = h->p;
    memset(out, 0, sizeof *out);
    out->n_envs = p.n_envs; out->jobs_max = p.jobs_max; out->machines_max = p.machines_max;
    out->mask_stride = p.mask_stride;
    out->action_mask = p.mask; out->real_obs = p.obs; out->solution = p.solution;
    out->host_mirror = h->host_block ? 1 : 0;
    out->mirror_actions = h->mirror_actions;
    out->scalar_stride = 16;   // reward / reward_raw / time / flags_done are fields of one 16-byte record per env
    out->reward = reinterpret_cast<float *>(p.scalars); out->reward_raw = p.scalars + 1;
    out->time = p.scalars + 2; out->flags_done = reinterpret_cast<uint32_t *>(p.scalars + 3);
    out->done = reinterpret_cast<uint8_t *>(p.scalars + 3);
    out->episode_count = p.episode_count; out->last_makespan = p.last_makespan; out->last_return = p.last_return;
    out->x_todo = p.x_todo; out->x_tufco = p.x_tufco; out->x_idle_last = p.x_idle_last;
    out->x_total_idle = p.x_total_idle; out->x_col4 = p.x_col4; out->x_tuam = p.x_tuam;
    out->x_legal = p.x_legal; out->x_blocked = p.x_blocked;
    return JSS_OK;
}

int jss_reset(jss_t *h, const uint8_t *env_mask_dev, void *stream) {
    int rc = check_ready(h);
    if (rc) return rc;
    JssLaunch a{};
    a.mode = JSS_MODE_RESET;
    a.env_mask = env_mask_dev;
    return launch_all(h, a, false, (cudaStream_t)stream);
}

int jss_step(jss_t *h, const int32_t *actions_dev, void *stream) {
    int rc = check_ready(h);
    if (rc) return rc;
    if (!actions_dev) return fail(h, JSS_ERR_INVALID, "jss_step: actions_dev is NULL");
    JssLaunch a{};
    a.mode = JSS_MODE_STEP;
    a.actions = actions_dev;
    return launch_all(h, a, false, (cudaStream_t)stream);
}

int jss_step_export(jss_t *h, const int32_t *actions_dev, void *stream) {
    int rc = check_ready(h);
    if (rc) return rc;
    if (!actions_dev) return fail(h, JSS_ERR_INVALID, "jss_step_export: actions_dev is NULL");
    if (h->gen) return fail(h, JSS_ERR_UNSUPPORTED, "jss_step_export: not available in generator mode");
    JssLaunch a{};
    a.mode = JSS_MODE_STEP;
    a.actions = actions_dev;
    a.export_after = 1;
    return launch_all(h, a, false, (cudaStream_t)stream);
}

int jss_step_sample(jss_t *h, const int32_t *actions_dev, int rule, int coin_mode, uint64_t seed,
                    uint64_t step_index, int32_t *next_actions_dev, void *stream) {
    int rc = check_ready(h);
    if (rc) return rc;
    if (!actions_dev || !next_actions_dev || rule < 0 || rule >= JSS_NUM_RULES ||
        (coin_mode != JSS_COIN_DEVICE && coin_mode != JSS_COIN_NEVER))
        return fail(h, JSS_ERR_INVALID, "jss_step_sample: bad arguments (rule %d, coin %d)", rule, coin_mode);
    JssLaunch a{};
    a.mode = JSS_MODE_STEP;
    a.actions = actions_dev;
    a.actions_out = next_actions_dev;
    a.rule = rule; a.coin_mode = coin_mode; a.seed = seed; a.step_index = step_index; a.cr_factor = h->cr_factor;
    a.hash_key = jss_hash_key(seed, step_index);
    return launch_all(h, a, false, (cudaStream_t)stream);
}

int jss_policy(jss_t *h, int rule, int coin_mode, uint64_t seed, uint64_t step_index, int32_t *actions_dev,
               void *stream) {
    int rc = check_ready(h);
    if (rc) return rc;
    if (!actions_dev || rule < 0 || rule >= JSS_NUM_RULES || (coin_mode != JSS_COIN_DEVICE && coin_mode != JSS_COIN_NEVER))
        return fail(h, JSS_ERR_INVALID, "jss_policy: bad arguments (rule %d, coin %d)", rule, coin_mode);
    JssLaunch a{};
    a.mode = JSS_MODE_POLICY;
    a.rule = rule; a.coin_mode = coin_mode; a.seed = seed; a.step_index = step_index; a.cr_factor = h->cr_factor;
    a.actions_out = actions_dev;
    return launch_all(h, a, rule_wants_rem(rule), (cudaStream_t)stream);
}

int jss_rollout(jss_t *h, int rule, uint64_t seed, uint64_t step_index, int n_steps, int write_obs, void *stream) {
    int rc = check_ready(h);
    if (rc) return rc;
    if (rule < 0 || rule >= JSS_NUM_RULES || n_steps < 0)
        return fail(h, JSS_ERR_INVALID, "jss_rollout: bad arguments (rule %d, n_steps %d)", rule, n_steps);
    JssLaunch a{};
    a.mode = JSS_MODE_ROLLOUT;
    a.rule = rule; a.coin_mode = JSS_COIN_DEVICE; a.seed = seed; a.step_index = step_index; a.cr_factor = h->cr_factor;
    a.n_steps = n_steps; a.write_obs = write_obs;
    return launch_all(h, a, rule_wants_rem(rule), (cudaStream_t)stream);
}

int jss_rollout_traj(jss_t *h, int rule, uint64_t seed, uint64_t step_index, int n_steps, float *traj_obs,
                     uint8_t *traj_mask, int32_t *traj_scalars, int32_t *traj_actions, void *stream) {
    int rc = check_ready(h);
    if (rc) return rc;
    if (rule < 0 || rule >= JSS_NUM_RULES || n_steps < 0 || !traj_obs || !traj_mask || !traj_scalars)
        return fail(h, JSS_ERR_INVALID, "jss_rollout_traj: bad arguments (rule %d, n_steps %d)", rule, n_steps);
    if ((int64_t)n_steps * h->n_envs >= INT32_MAX)
        return fail(h, JSS_ERR_UNSUPPORTED, "jss_rollout_traj: n_steps * n_envs must stay below 2^31");
    JssLaunch a{};
    a.mode = JSS_MODE_ROLLOUT;
    a.rule = rule; a.coin_mode = JSS_COIN_DEVICE; a.seed = seed; a.step_index = step_index; a.cr_factor = h->cr_factor;
    a.n_steps = n_steps; a.write_obs = 1;
    a.traj_obs = traj_obs; a.traj_mask = traj_mask; a.traj_scalars = traj_scalars; a.traj_actions = traj_actions;
    return launch_all(h, a, rule_wants_rem(rule), (cudaStream_t)stream);
}

int jss_step_host(jss_t *h, const int32_t *actions_host, uint8_t *mask_host, float *obs_host,
                  int32_t *scalars_host, void *stream) {
    int rc = check_ready(h);
    if (rc) return rc;
    if (!actions_host) return fail(h, JSS_ERR_INVALID, "jss_step_host: actions_host is NULL");
    cudaStream_t st = (cudaStream_t)stream;
    const JssParams &p = h->p;
    const size_t N = (size_t)p.n_envs;
    JSS_CUDA(h, cudaMemcpyAsync(h->dev_actions, actions_host, N * 4, cudaMemcpyHostToDevice, st));
    rc = jss_step(h, h->dev_actions, stream);
    if (rc) return rc;
    // contiguous DMA only: host rows keep the device pitches (mask rows: mask_stride bytes,
    // scalar records: 16 bytes) -- pitched 2-D copies of 65 536 tiny rows are several times slower
    if (mask_host)
        JSS_CUDA(h, cudaMemcpyAsync(mask_host, p.mask, N * p.mask_stride, cudaMemcpyDeviceToHost, st));
    if (obs_host)
        JSS_CUDA(h, cudaMemcpyAsync(obs_host, p.obs, N * p.jobs_max * 7 * 4, cudaMemcpyDeviceToHost, st));
    if (scalars_host) JSS_CUDA(h, cudaMemcpyAsync(scalars_host, p.scalars, N * 16, cudaMemcpyDeviceToHost, st));
    JSS_CUDA(h, cudaStreamSynchronize(st));
    return JSS_OK;
}

namespace {
// obs_host != NULL: envs [0, n_dma) ship their observation as fp32 rows by DMA (n_dma < 0: all of them);
// wire_host != NULL: envs [max(n_dma, 0), N) ship packed integer rows.
int host_step_begin_impl(jss_t *h, const int32_t *actions_host, uint8_t *mask_host, float *obs_host, uint8_t *wire_host,
                         int32_t *scalars_host, void *after_stream, int n_dma = -1) {
    int rc = check_ready(h);
    if (rc) return rc;
    if (!actions_host) return fail(h, JSS_ERR_INVALID, "jss_host_step_begin: actions_host is NULL");
    if (wire_host && h->gen)   // the host expansion holds per-instance divisors
        return fail(h, JSS_ERR_UNSUPPORTED, "packed / hybrid host steps are not available in generator mode");
    const JssParams &p = h->p;
    const size_t N = (size_t)p.n_envs;
    const size_t n_fp32 = obs_host ? (n_dma < 0 ? N : std::min<size_t>((size_t)n_dma, N)) : 0;     // envs [0, n_fp32): fp32 by DMA
    const size_t obs_bytes = n_fp32 * p.jobs_max * 7 * 4;
    if (!h->pipe_ready) {
        JSS_CUDA(h, cudaStreamCreateWithFlags(&h->s_compute, cudaStreamNonBlocking));
        JSS_CUDA(h, cudaStreamCreateWithFlags(&h->s_copy, cudaStreamNonBlocking));
        JSS_CUDA(h, cudaEventCreateWithFlags(&h->ev_mask, cudaEventDisableTiming));
        JSS_CUDA(h, cudaEventCreateWithFlags(&h->ev_staged, cudaEventDisableTiming));
        JSS_CUDA(h, cudaEventCreateWithFlags(&h->ev_wire, cudaEventDisableTiming));
        for (int k = 0; k < 2; k++) {
            JSS_CUDA(h, cudaEventCreateWithFlags(&h->ev_obs[k], cudaEventDisableTiming));
            JSS_CUDA(h, cudaEventRecord(h->ev_obs[k], h->s_copy));
        }
        h->pipe_ready = true;
    }
    if (obs_host && !h->obs_staging && (rc = dev_alloc(h, &h->obs_staging, N * p.jobs_max * 7, false))) return rc;
    if (wire_host && !h->wire[0]) {
        // 16-byte multiple with >= 6 bytes of slack behind the last record (the host expansion loads 16 bytes per job)
        h->wire_stride = round_up(JSS_WIRE_JOB_BYTES * p.jobs_max + 6, 16);
        for (int k = 0; k < 2; k++)
            if ((rc = dev_alloc(h, &h->wire[k], N * (size_t)h->wire_stride))) return rc;
    }
    cudaStream_t sc = h->s_compute;
    // order the pipeline after whatever the caller enqueued on its own stream (reset, device-side steps ...)
    JSS_CUDA(h, cudaEventRecord(h->ev_staged, (cudaStream_t)after_stream));
    JSS_CUDA(h, cudaStreamWaitEvent(sc, h->ev_staged, 0));
    JSS_CUDA(h, cudaMemcpyAsync(h->dev_actions, actions_host, N * 4, cudaMemcpyHostToDevice, sc));
    rc = jss_step(h, h->dev_actions, (void *)sc);
    if (rc) return rc;
    // the small results first: a host policy only needs the mask.  If the host buffers are pinned
    // (device-mappable) the SMs write them directly; otherwise fall back to the copy engine.
    auto small_d2h = [&](void *dst_host, const void *src_dev, size_t bytes) -> int {
        void *mapped = nullptr;
        if ((bytes & 15) == 0 && cudaHostGetDevicePointer(&mapped, dst_host, 0) == cudaSuccess && mapped) {
            const size_t n16 = bytes / 16;
            const int blocks = (int)std::min<size_t>((n16 + 255) / 256, (size_t)h->sm_count * 8);
            JSS_LAUNCH(jss_copy16_kernel, blocks, 256, 0, sc, (uint4 *)mapped, (const uint4 *)src_dev, n16);
            JSS_CUDA(h, cudaGetLastError());
            h->launches += 1;
        } else {
            (void)cudaGetLastError();
            JSS_CUDA(h, cudaMemcpyAsync(dst_host, src_dev, bytes, cudaMemcpyDeviceToHost, sc));
        }
        return JSS_OK;
    };
    if (mask_host && (rc = small_d2h(mask_host, p.mask, N * p.mask_stride))) return rc;
    if (scalars_host && (rc = small_d2h(scalars_host, p.scalars, N * 16))) return rc;
    JSS_CUDA(h, cudaEventRecord(h->ev_mask, sc));
    const int prev = h->pipe_cur;
    h->pipe_cur ^= 1;
    if (obs_bytes) {
        // observation: device-side staging copy (so the next step may overwrite real_obs), then the
        // 2.9 KB/env PCIe transfer on its own stream, overlapping the host policy and the next launch
        JSS_CUDA(h, cudaStreamWaitEvent(sc, h->ev_obs[prev], 0));      // previous D2H has drained the staging copy
        JSS_CUDA(h, cudaMemcpyAsync(h->obs_staging, p.obs, obs_bytes, cudaMemcpyDeviceToDevice, sc));
    }
    if (wire_host && n_fp32 < N) {
        // packed rows: 10 bytes per job instead of 28; two device buffers alternate, so this pack only has to wait
        // for the D2H that read the same buffer two begins ago
        JSS_CUDA(h, cudaStreamWaitEvent(sc, h->ev_obs[h->pipe_cur], 0));
        JssLaunch a{};
        a.mode = JSS_MODE_PACK;
        a.wire = h->wire[h->pipe_cur];
        a.wire_stride = (int32_t)h->wire_stride;
        if ((rc = launch_all(h, a, false, sc))) return rc;
    }
    // the copy stream never runs ahead of the step (also when nothing large is copied: JSS_WAIT_OBS is the barrier
    // callers take before going back to the stream-ordered entry points)
    JSS_CUDA(h, cudaEventRecord(h->ev_staged, sc));
    JSS_CUDA(h, cudaStreamWaitEvent(h->s_copy, h->ev_staged, 0));
    if (wire_host && n_fp32 < N) {       // the packed rows first: the host has to expand them, the fp32 rows are final
        const size_t off = n_fp32 * (size_t)h->wire_stride;
        JSS_CUDA(h, cudaMemcpyAsync(wire_host + off, h->wire[h->pipe_cur] + off, (N - n_fp32) * (size_t)h->wire_stride,
                                    cudaMemcpyDeviceToHost, h->s_copy));
        JSS_CUDA(h, cudaEventRecord(h->ev_wire, h->s_copy));
    }
    if (obs_bytes)
        JSS_CUDA(h, cudaMemcpyAsync(obs_host, h->obs_staging, obs_bytes, cudaMemcpyDeviceToHost, h->s_copy));
    JSS_CUDA(h, cudaEventRecord(h->ev_obs[h->pipe_cur], h->s_copy));
    return JSS_OK;
}
}  // namespace

int jss_host_step_begin(jss_t *h, const int32_t *actions_host, uint8_t *mask_host, float *obs_host,
                        int32_t *scalars_host, void *after_stream) {
    return host_step_begin_impl(h, actions_host, mask_host, obs_host, nullptr, scalars_host, after_stream);
}

int jss_host_step_begin_packed(jss_t *h, const int32_t *actions_host, uint8_t *mask_host, uint8_t *wire_host,
                               int32_t *scalars_host, void *after_stream) {
    if (!wire_host || !scalars_host)
        return fail(h, JSS_ERR_INVALID, "jss_host_step_begin_packed: wire_host and scalars_host are required");
    return host_step_begin_impl(h, actions_host, mask_host, nullptr, wire_host, scalars_host, after_stream);
}

int jss_host_step_begin_hybrid(jss_t *h, const int32_t *actions_host, uint8_t *mask_host, uint8_t *wire_host,
                               float *obs_host, int n_dma, int32_t *scalars_host, void *after_stream) {
    if (!wire_host || !obs_host || !scalars_host || n_dma < 0)
        return fail(h, JSS_ERR_INVALID, "jss_host_step_begin_hybrid: wire_host, obs_host, scalars_host and n_dma >= 0 are required");
    return host_step_begin_impl(h, actions_host, mask_host, obs_host, wire_host, scalars_host, after_stream, n_dma);
}

int64_t jss_host_wire_stride(jss_t *h) {
    if (!h || !h->assigned) return JSS_ERR_STATE;
    return round_up(JSS_WIRE_JOB_BYTES * h->p.jobs_max + 6, 16);
}

int jss_host_expand_obs(jss_t *h, const uint8_t *wire_host, const int32_t *scalars_host, float *obs_host) {
    return jss_host_expand_obs_range(h, wire_host, scalars_host, obs_host, 0, h ? h->n_envs : 0);
}

int jss_host_expand_obs_range(jss_t *h, const uint8_t *wire_host, const int32_t *scalars_host, float *obs_host,
                              int env_begin, int env_end) {
    if (!h || !h->assigned) return fail(h, JSS_ERR_STATE, "jss_host_expand_obs: jss_assign must be called first");
    if (!wire_host || !scalars_host || !obs_host || env_begin < 0 || env_end > h->n_envs || env_begin > env_end)
        return fail(h, JSS_ERR_INVALID, "jss_host_expand_obs: bad arguments");
    if (h->gen) return fail(h, JSS_ERR_UNSUPPORTED, "jss_host_expand_obs: not available in generator mode");
    std::vector<JssHostInst> hi(h->insts.size());
    for (size_t k = 0; k < h->insts.size(); k++)
        hi[k] = JssHostInst{h->insts[k].J, h->insts[k].M, h->insts[k].max_time_op, h->insts[k].max_time_jobs,
                            h->insts[k].sum_op, h->insts[k].len.data()};
    JssHostExpandArgs a{wire_host, jss_host_wire_stride(h), scalars_host, h->env_inst.data(), hi.data(), obs_host,
                        h->p.jobs_max, env_begin, env_end};
    jss_host_expand_impl(&a);
    return JSS_OK;
}

int jss_host_configure(int threads, int bind_numa_of_device) {
    std::vector<int> cpus;
#ifndef JSS_EMU
    if (bind_numa_of_device >= 0) {
        // CPUs of the NUMA node the GPU hangs off (pinned buffers and the expansion threads stay local to it)
        char bus[32] = {0};
        if (cudaDeviceGetPCIBusId(bus, sizeof bus, bind_numa_of_device) == cudaSuccess) {
            for (char *c = bus; *c; c++) *c = (char)tolower(*c);
            char path[160];
            snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/numa_node", bus);
            int node = -1;
            if (FILE *f = fopen(path, "r")) { if (fscanf(f, "%d", &node) != 1) node = -1; fclose(f); }
            if (node >= 0) {
                snprintf(path, sizeof path, "/sys/devices/system/node/node%d/cpulist", node);
                if (FILE *f = fopen(path, "r")) {
                    int a = 0, b = 0;
                    char sep = 0;
                    cpu_set_t allowed;
                    const bool have = sched_getaffinity(0, sizeof allowed, &allowed) == 0;
                    while (fscanf(f, "%d", &a) == 1) {
                        b = a;
                        if (fscanf(f, "%c", &sep) == 1 && sep == '-') { if (fscanf(f, "%d", &b) != 1) b = a; if (fscanf(f, "%c", &sep) != 1) sep = 0; }
                        for (int c = a; c <= b; c++)
                            if (!have || CPU_ISSET(c, &allowed)) cpus.push_back(c);
                        if (sep != ',') break;
                    }
                    fclose(f);
                }
            }
        }
        (void)cudaGetLastError();
    }
#else
    (void)bind_numa_of_device;
#endif
    jss_host_pool_configure(threads, cpus.data(), (int)cpus.size());
    return (int)cpus.size();
}

int jss_host_threads(void) { return jss_host_pool_size(); }

int jss_host_set_simd(int level) { jss_host_simd_cap(level); return JSS_OK; }

int jss_host_wait(jss_t *h, int what) {
    int rc = check_ready(h);
    if (rc) return rc;
    if (!h->pipe_ready) return fail(h, JSS_ERR_STATE, "jss_host_wait: no jss_host_step_begin in flight");
    if (what == JSS_WAIT_MASK) JSS_CUDA(h, cudaEventSynchronize(h->ev_mask));
    else if (what == JSS_WAIT_OBS) JSS_CUDA(h, cudaEventSynchronize(h->ev_obs[h->pipe_cur]));
    else if (what == JSS_WAIT_OBS_PREV) JSS_CUDA(h, cudaEventSynchronize(h->ev_obs[h->pipe_cur ^ 1]));
    else if (what == JSS_WAIT_WIRE) JSS_CUDA(h, cudaEventSynchronize(h->ev_wire));
    else return fail(h, JSS_ERR_INVALID, "jss_host_wait: unknown selector %d", what);
    return JSS_OK;
}

int jss_stats(jss_t *h, int64_t *out_host, void *stream) {
    int rc = check_ready(h);
    if (rc) return rc;
    if (!out_host) return fail(h, JSS_ERR_INVALID, "jss_stats: out_host is NULL");
    cudaStream_t st = (cudaStream_t)stream;
    unsigned long long init[JSS_STATS_LEN] = {0, 0, 0, ~0ull, 0, 0, 0, 0};
    JSS_CUDA(h, cudaMemcpyAsync(h->d_stats, init, sizeof init, cudaMemcpyHostToDevice, st));
    const int threads = 256;
    const int blocks = std::min((h->n_envs + threads - 1) / threads, h->sm_count * 4);
    JSS_LAUNCH(jss_stats_kernel, blocks, threads, 0, st, h->p, h->d_stats);
    JSS_CUDA(h, cudaGetLastError());
    h->launches += 1;
    unsigned long long res[JSS_STATS_LEN];
    JSS_CUDA(h, cudaMemcpyAsync(res, h->d_stats, sizeof res, cudaMemcpyDeviceToHost, st));
    JSS_CUDA(h, cudaStreamSynchronize(st));
    for (int i = 0; i < JSS_STATS_LEN; i++) out_host[i] = (int64_t)res[i];
    if (res[3] == ~0ull) out_host[3] = INT64_MAX;
    return JSS_OK;
}

int jss_export_state(jss_t *h, void *stream) {
    int rc = check_ready(h);
    if (rc) return rc;
    JssLaunch a{};
    a.mode = JSS_MODE_EXPORT;
    return launch_all(h, a, false, (cudaStream_t)stream);
}

int jss_import_state(jss_t *h, const uint8_t *env_mask_dev, void *stream) {
    int rc = check_ready(h);
    if (rc) return rc;
    if (h->gen)   // a restored state would not match the instance the env has drawn since
        return fail(h, JSS_ERR_UNSUPPORTED, "jss_import_state: not available in generator mode");
    JssLaunch a{};
    a.mode = JSS_MODE_IMPORT;
    a.env_mask = env_mask_dev;
    return launch_all(h, a, false, (cudaStream_t)stream);
}

int jss_host_masked_random(const uint8_t *mask_host, int n, int width, int64_t row_stride, uint64_t seed,
                           uint64_t env_id_base, uint64_t step_index, int32_t *actions_host) {
    if (!mask_host || !actions_host || n < 0 || width <= 0 || row_stride < width) return JSS_ERR_INVALID;
    jss_host_masked_random_impl(mask_host, n, width, row_stride, seed, env_id_base, step_index, actions_host);   // persistent pool
    return JSS_OK;
}

}  // extern "C"
