// jss_host.cpp -- host-side helpers of the C-ABI (plain C++, compiled by the host compiler):
//   * a persistent worker pool (sized to the CPUs this process may use, optionally bound to the
//     NUMA node of its GPU) shared by the helpers below;
//   * jss_host_masked_random(): the device sampler's draw from a HOST mask (host-side agents, tests, e2e bench);
//   * the expansion of the packed observation wire format (jss_host_step_begin_packed) into the
//     reference's float observation (JSSEnv/envs/jss_env.py:102-134) -- exact: the wire carries the integer
//     numerators, the quotients are IEEE fp32 divisions, i.e. the same correctly rounded values the device
//     kernels write to real_obs (tools/check_div.c).
// Nothing here computes environment transitions: there is no CPU implementation of the environment.
#include "jss_host.h"

#include <sched.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <math.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include <vector>

#if defined(__x86_64__)
#include <immintrin.h>
#define JSS_HAVE_AVX2_TARGET 1
#endif

#include "jss_rng.h"

namespace {

// ---- CPUs this process may use: min(affinity mask, cgroup quota) ---------------------------------
int usable_cpus() {
    int n = (int)std::max(1u, std::thread::hardware_concurrency());
    cpu_set_t set;
    if (sched_getaffinity(0, sizeof set, &set) == 0) n = std::min(n, std::max(1, CPU_COUNT(&set)));
    if (FILE *f = fopen("/sys/fs/cgroup/cpu.max", "r")) {          // cgroup v2 quota, if any
        long long q = 0, per = 0;
        if (fscanf(f, "%lld %lld", &q, &per) == 2 && q > 0 && per > 0) n = std::min<long long>(n, (q + per - 1) / per);
        fclose(f);
    }
    return std::max(1, n);
}

// ---- persistent pool -------------------------------------------------------------------------------
// parallel_for(n_items, grain, fn): fn(begin, end) on chunks of `grain` items handed out by an atomic
// cursor; the calling thread works too.  Workers are created once and sleep on a condition variable.
class Pool {
  public:
    static Pool &get() { static Pool p; return p; }

    void configure(int threads, const std::vector<int> &cpus) {
        std::lock_guard<std::mutex> g(api_);
        stop();
        want_ = threads;
        cpus_ = cpus;
    }
    int size() {
        std::lock_guard<std::mutex> g(api_);
        ensure();
        return (int)workers_.size() + 1;
    }
    void parallel_for(int64_t n, int64_t grain, const std::function<void(int64_t, int64_t)> &fn) {
        if (n <= 0) return;
        std::lock_guard<std::mutex> g(api_);                  // one parallel region at a time
        ensure();
        if (workers_.empty() || n <= grain) { fn(0, n); return; }
        {
            std::lock_guard<std::mutex> lk(m_);
            fn_ = &fn; n_ = n; grain_ = grain; cursor_.store(0); pending_ = (int)workers_.size(); gen_++;
        }
        cv_.notify_all();
        work();
        std::unique_lock<std::mutex> lk(m_);
        done_cv_.wait(lk, [&] { return pending_ == 0; });
        fn_ = nullptr;
    }
    ~Pool() { stop(); }

  private:
    void work() {
        for (;;) {
            const int64_t b = cursor_.fetch_add(grain_);
            if (b >= n_) break;
            (*fn_)(b, std::min(n_, b + grain_));
        }
    }
    void ensure() {
        if (started_) return;
        started_ = true;
        int t = want_ > 0 ? want_ : usable_cpus();
        if (const char *lw = getenv("LOCAL_WORLD_SIZE")) {       // torchrun: share the host between the local ranks
            const int k = atoi(lw);
            if (want_ <= 0 && k > 1) t = std::max(1, t / k);
        }
        // CPU list the workers are spread over: the NUMA node's CPUs given to configure(), else the affinity mask
        std::vector<int> list = cpus_;
        if (list.empty()) {
            cpu_set_t set;
            if (sched_getaffinity(0, sizeof set, &set) == 0)
                for (int c = 0; c < CPU_SETSIZE; c++)
                    if (CPU_ISSET(c, &set)) list.push_back(c);
        }
        // One CPU per worker (default) is the fastest layout on a quiet host (e2e 31 M vs 25 M env-steps/s with workers only
        // confined to the node), but on a shared box a busy CPU in the list stalls every parallel region; JSS_HOST_PIN=0
        // confines the workers to the CPU list (the GPU's NUMA node) and lets the scheduler place them.  bench.py
        // calibrates both layouts on the box it runs on.
        const char *pin_env = getenv("JSS_HOST_PIN");
        const bool pin = !(pin_env && pin_env[0] == '0') && !list.empty() && t <= (int)list.size();
        int offset = 0;
        if (const char *lr = getenv("LOCAL_RANK")) offset = atoi(lr) * t;      // local ranks take disjoint slices
        // gen_ survives configure(): a new worker starts at the current generation, so that it answers only regions issued
        // after it exists.  A worker starting below it would run a stale region and decrement pending_ twice, and
        // parallel_for could return while another worker is still inside fn.  Read under api_, the only lock gen_ changes under.
        const uint64_t start = gen_;
        for (int i = 1; i < t; i++) {
            const int cpu = pin ? list[(size_t)(offset + i) % list.size()] : -1;
            workers_.emplace_back([this, cpu, list, start] {
                cpu_set_t set; CPU_ZERO(&set);
                if (cpu >= 0) CPU_SET(cpu, &set);
                else for (int c : list) CPU_SET(c, &set);
                if (cpu >= 0 || !cpus_.empty()) sched_setaffinity(0, sizeof set, &set);
                uint64_t seen = start;
                for (;;) {
                    {
                        std::unique_lock<std::mutex> lk(m_);
                        cv_.wait(lk, [&] { return quit_ || gen_ != seen; });
                        if (quit_) return;
                        seen = gen_;
                    }
                    work();
                    std::lock_guard<std::mutex> lk(m_);
                    if (--pending_ == 0) done_cv_.notify_one();
                }
            });
        }
    }
    void stop() {
        {
            std::lock_guard<std::mutex> lk(m_);
            quit_ = true;
        }
        cv_.notify_all();
        for (auto &t : workers_) t.join();
        workers_.clear();
        quit_ = false; started_ = false;
    }

    std::mutex api_, m_;
    std::condition_variable cv_, done_cv_;
    std::vector<std::thread> workers_;
    std::vector<int> cpus_;
    const std::function<void(int64_t, int64_t)> *fn_ = nullptr;
    std::atomic<int64_t> cursor_{0};
    int64_t n_ = 0, grain_ = 1;
    int pending_ = 0, want_ = 0;
    uint64_t gen_ = 0;
    bool quit_ = false, started_ = false;
};

// ---- packed observation -> float rows ----------------------------------------------------------------
// Wire record of one job (JSS_WIRE_JOB_BYTES = 10, little endian):
//   bytes 0..3  w0 = legal | tufco << 1 | todo << 12 | col4 << 18      (1 + 11 + 6 + 11 bits)
//   bytes 4..6  idle_time_jobs_last_op   (24 bits; the makespan bound J*M*2047 < 2^24)
//   bytes 7..9  total_idle_time_jobs     (24 bits)
// total_perform_op_time_jobs (column 3) is not shipped: it equals t - total_idle while the job is unfinished and
// jobs_length[j] afterwards; t travels in the env's scalar record.
struct Cols {                  // per output column: divisor 1, max_time_op, M, max_time_jobs, max_time_op, sum_op, sum_op
    float d[16], r[16];        // d = divisor, r = RN(1 / divisor); the 7-column pattern twice (two jobs per 512-bit vector)
};

// The device's quotient (jss_div in jss_device.cuh): q = RN(x * r); e = x - q * d (exact, FMA); q' = RN(q + e * r).
// Same operations in the same order here, so the expanded observation equals real_obs bit for bit.
inline float markstein(float x, float d, float r) {
    const float q = x * r;
    const float e = fmaf(-q, d, x);
    return fmaf(e, r, q);
}

inline void expand_job_scalar(const uint8_t *rec, int t, int M, int len, const Cols &c, float *out) {
    uint32_t w0;
    memcpy(&w0, rec, 4);
    const int idle = rec[4] | (rec[5] << 8) | (rec[6] << 16), total = rec[7] | (rec[8] << 8) | (rec[9] << 16);
    const int todo = (int)((w0 >> 12) & 63u);
    const int perf = todo < M ? t - total : len;
    out[0] = (float)(w0 & 1u);
    out[1] = markstein((float)((w0 >> 1) & 2047u), c.d[1], c.r[1]);
    out[2] = markstein((float)todo, c.d[2], c.r[2]);
    out[3] = markstein((float)perf, c.d[3], c.r[3]);
    out[4] = markstein((float)((w0 >> 18) & 2047u), c.d[4], c.r[4]);
    out[5] = markstein((float)idle, c.d[5], c.r[5]);
    out[6] = markstein((float)total, c.d[6], c.r[6]);
}

void expand_env_scalar(const uint8_t *row, int J, int M, int t, const int32_t *len, const Cols &c, float *out) {
    for (int j = 0; j < J; j++) expand_job_scalar(row + (size_t)j * JSS_WIRE_JOB_BYTES, t, M, len[j], c, out + 7 * j);
}

#ifdef JSS_HAVE_AVX2_TARGET
// one job per iteration: 16-byte load, byte shuffle to dwords, per-lane shift + mask, convert, divide
__attribute__((target("avx2,fma"))) void expand_env_avx2(const uint8_t *row, int J, int M, int t, const int32_t *len,
                                                    const Cols &c, float *out) {
    const __m128i shuf = _mm_setr_epi8(0, 1, 2, 3, 4, 5, 6, (char)0x80, 7, 8, 9, (char)0x80, (char)0x80, (char)0x80,
                                       (char)0x80, (char)0x80);                    // -> [w0, idle, total, 0]
    const __m256i pick = _mm256_setr_epi32(0, 0, 0, 3, 0, 1, 2, 3);                // lane 3 (perf) is patched in below
    const __m256i shift = _mm256_setr_epi32(0, 1, 12, 0, 18, 0, 0, 0);
    const __m256i mask = _mm256_setr_epi32(1, 2047, 63, -1, 2047, 0xFFFFFF, 0xFFFFFF, 0);
    const __m256 div = _mm256_loadu_ps(c.d), rcp = _mm256_loadu_ps(c.r);
    const __m256i store7 = _mm256_setr_epi32(-1, -1, -1, -1, -1, -1, -1, 0);
    for (int j = 0; j < J; j++) {
        const __m128i raw = _mm_loadu_si128(reinterpret_cast<const __m128i *>(row + (size_t)j * JSS_WIRE_JOB_BYTES));
        __m128i d4 = _mm_shuffle_epi8(raw, shuf);
        const uint32_t w0 = (uint32_t)_mm_cvtsi128_si32(d4);
        const int total = _mm_extract_epi32(d4, 2);
        const int todo = (int)((w0 >> 12) & 63u);
        d4 = _mm_insert_epi32(d4, todo < M ? t - total : len[j], 3);
        __m256i v = _mm256_permutevar8x32_epi32(_mm256_castsi128_si256(d4), pick);
        v = _mm256_and_si256(_mm256_srlv_epi32(v, shift), mask);
        const __m256 x = _mm256_cvtepi32_ps(v);
        __m256 q = _mm256_mul_ps(x, rcp);
        q = _mm256_fmadd_ps(_mm256_fnmadd_ps(q, div, x), rcp, q);       // Markstein, as on the device
        if (j + 1 < J) _mm256_storeu_ps(out + 7 * j, q);        // the 8th float is overwritten by the next job
        else _mm256_maskstore_ps(out + 7 * j, store7, q);
    }
}
// two jobs (14 floats) per 512-bit vector
__attribute__((target("avx512f,avx512bw,avx512vl,avx512dq"))) void expand_env_avx512(const uint8_t *row, int J, int M, int t,
                                                                                   const int32_t *len, const Cols &c, float *out) {
    const __m128i shuf = _mm_setr_epi8(0, 1, 2, 3, 4, 5, 6, (char)0x80, 7, 8, 9, (char)0x80, (char)0x80, (char)0x80,
                                       (char)0x80, (char)0x80);                    // -> [w0, idle, total, 0]
    // source dwords: job A = 0..2, job B = 4..6.  Output lanes: A = 0..6, B = 7..13.
    const __m512i pick = _mm512_setr_epi32(0, 0, 0, 2, 0, 1, 2, 4, 4, 4, 6, 4, 5, 6, 0, 0);
    const __m512i shift = _mm512_setr_epi32(0, 1, 12, 0, 18, 0, 0, 0, 1, 12, 0, 18, 0, 0, 0, 0);
    const __m512i mask = _mm512_setr_epi32(1, 2047, 63, 0xFFFFFF, 2047, 0xFFFFFF, 0xFFFFFF, 1, 2047, 63, 0xFFFFFF, 2047,
                                           0xFFFFFF, 0xFFFFFF, 0, 0);
    const __m512i lenpick = _mm512_setr_epi32(0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 0, 0, 0, 0, 0);   // lane 3 <- len[j], lane 10 <- len[j+1]
    const __m512 div = _mm512_loadu_ps(c.d), rcp = _mm512_loadu_ps(c.r);
    const __m512i tv = _mm512_set1_epi32(t), mv = _mm512_set1_epi32(M);
    const __mmask16 todo_lanes = (1u << 2) | (1u << 9), perf_lanes = (1u << 3) | (1u << 10);
    int j = 0;
    for (; j + 2 <= J; j += 2) {
        const uint8_t *rec = row + (size_t)j * JSS_WIRE_JOB_BYTES;
        const __m128i a = _mm_shuffle_epi8(_mm_loadu_si128(reinterpret_cast<const __m128i *>(rec)), shuf);
        const __m128i b = _mm_shuffle_epi8(_mm_loadu_si128(reinterpret_cast<const __m128i *>(rec + JSS_WIRE_JOB_BYTES)), shuf);
        const __m512i src = _mm512_castsi256_si512(_mm256_inserti128_si256(_mm256_castsi128_si256(a), b, 1));
        __m512i v = _mm512_and_si512(_mm512_srlv_epi32(_mm512_permutexvar_epi32(pick, src), shift), mask);
        // column 3: t - total_idle while the job is unfinished (todo < M), jobs_length afterwards
        const __mmask16 unfinished = (__mmask16)(_mm512_mask_cmplt_epi32_mask(todo_lanes, v, mv) << 1);
        const __m512i lens = _mm512_permutexvar_epi32(lenpick, _mm512_castsi128_si512(_mm_loadl_epi64(reinterpret_cast<const __m128i *>(len + j))));
        const __m512i perf = _mm512_mask_mov_epi32(lens, unfinished, _mm512_sub_epi32(tv, v));
        v = _mm512_mask_mov_epi32(v, perf_lanes, perf);
        const __m512 x = _mm512_cvtepi32_ps(v);
        __m512 q = _mm512_mul_ps(x, rcp);
        q = _mm512_fmadd_ps(_mm512_fnmadd_ps(q, div, x), rcp, q);       // Markstein, as on the device
        _mm512_mask_storeu_ps(out + 7 * j, (__mmask16)0x3FFF, q);
    }
    for (; j < J; j++) expand_job_scalar(row + (size_t)j * JSS_WIRE_JOB_BYTES, t, M, len[j], c, out + 7 * j);
}
std::atomic<int> g_simd_cap{2};   // tests lower this to exercise the narrower code paths (jss_host_set_simd)
bool have_avx512() {
    static const bool v = __builtin_cpu_supports("avx512f") && __builtin_cpu_supports("avx512bw") &&
                          __builtin_cpu_supports("avx512vl") && __builtin_cpu_supports("avx512dq");
    return v && g_simd_cap.load() >= 2;
}

// dst and n need no alignment; cache-bypassing stores for the 64-byte-aligned body (the expanded batch is
// far larger than the caches and is consumed by somebody else)
__attribute__((target("avx2"))) void stream_copy(float *dst, const float *src, size_t n) {
    static const bool nt = !(getenv("JSS_HOST_NT") && getenv("JSS_HOST_NT")[0] == '0');   // experiments: regular stores
    if (!nt) { memcpy(dst, src, n * sizeof(float)); return; }
    size_t i = 0;
    while (i < n && (reinterpret_cast<uintptr_t>(dst + i) & 63u)) { dst[i] = src[i]; i++; }
    for (; i + 16 <= n; i += 16) {
        _mm256_stream_ps(dst + i, _mm256_loadu_ps(src + i));
        _mm256_stream_ps(dst + i + 8, _mm256_loadu_ps(src + i + 8));
    }
    for (; i < n; i++) dst[i] = src[i];
}
bool have_avx2() {
    static const bool v = __builtin_cpu_supports("avx2") && __builtin_cpu_supports("fma");
    return v && g_simd_cap.load() >= 1;
}
#else
std::atomic<int> g_simd_cap{0};
bool have_avx2() { return false; }
bool have_avx512() { return false; }
#endif

}  // namespace

int jss_host_pool_configure(int threads, const int *cpus, int n_cpus) {
    std::vector<int> v;
    for (int i = 0; i < n_cpus; i++) v.push_back(cpus[i]);
    Pool::get().configure(threads, v);
    return 0;
}

int jss_host_pool_size(void) { return Pool::get().size(); }

void jss_host_simd_cap(int level) { g_simd_cap.store(level); }

void jss_host_parallel_for(int64_t n, int64_t grain, void (*fn)(int64_t, int64_t, void *), void *ctx) {
    Pool::get().parallel_for(n, grain, [&](int64_t b, int64_t e) { fn(b, e, ctx); });
}

#ifdef JSS_HAVE_AVX2_TARGET
// one mask row: count the set bytes and return the index of the r-th one, 32 bytes at a time (the row may be read up
// to the next multiple of 32 past `width` only if that stays inside the row stride)
__attribute__((target("avx2,bmi2,popcnt"))) int pick_row_avx2(const uint8_t *row, int width, uint32_t h) {
    uint32_t bits[8];                                     // width <= 129 -> at most 5 words of 32 mask bytes
    const int nw = (width + 31) >> 5;
    const __m256i zero = _mm256_setzero_si256();
    int cnt = 0;
    for (int w = 0; w < nw; w++) {
        const int left = width - 32 * w;
        __m256i v;
        if (left >= 32) v = _mm256_loadu_si256(reinterpret_cast<const __m256i *>(row + 32 * w));
        else {
            alignas(32) uint8_t tmp[32] = {0};
            memcpy(tmp, row + 32 * w, (size_t)left);
            v = _mm256_load_si256(reinterpret_cast<const __m256i *>(tmp));
        }
        bits[w] = ~(uint32_t)_mm256_movemask_epi8(_mm256_cmpeq_epi8(v, zero));
        cnt += __builtin_popcount(bits[w]);
    }
    if (cnt == 0) return -1;
    uint32_t r = jss_pick(h, (uint32_t)cnt);
    for (int w = 0; w < nw; w++) {
        const uint32_t c = (uint32_t)__builtin_popcount(bits[w]);
        if (r < c) return 32 * w + (int)__builtin_ctz(_pdep_u32(1u << r, bits[w]));
        r -= c;
    }
    return -1;
}
bool have_bmi2() { static const bool v = __builtin_cpu_supports("avx2") && __builtin_cpu_supports("bmi2"); return v; }
#endif

void jss_host_masked_random_impl(const uint8_t *mask_host, int n, int width, int64_t row_stride, uint64_t seed,
                                 uint64_t env_id_base, uint64_t step_index, int32_t *actions_host) {
    auto work = [&](int64_t lo, int64_t hi) {
        for (int64_t e = lo; e < hi; e++) {
            const uint8_t *row = mask_host + (size_t)e * (size_t)row_stride;
            const uint32_t hsh = jss_hash3(seed, env_id_base + (uint64_t)e, step_index);
#ifdef JSS_HAVE_AVX2_TARGET
            if (width <= 256 && have_bmi2() && g_simd_cap.load(std::memory_order_relaxed) >= 1) {
                actions_host[e] = pick_row_avx2(row, width, hsh);
                continue;
            }
#endif
            int cnt = 0;
            for (int i = 0; i < width; i++) cnt += row[i] != 0;
            int act = -1;   // JSS_ACTION_SKIP
            if (cnt > 0) {
                uint32_t r = jss_pick(hsh, (uint32_t)cnt);
                for (int i = 0; i < width; i++)
                    if (row[i]) { if (r == 0) { act = i; break; } r--; }
            }
            actions_host[e] = act;
        }
    };
    if ((int64_t)n * width < (1 << 16)) { work(0, n); return; }
    Pool::get().parallel_for(n, 1024, work);
}

void jss_host_expand_impl(const JssHostExpandArgs *a) {
    auto work = [&](int64_t lo, int64_t hi) {
        std::vector<float> stage((size_t)a->jobs_max * 7 + 8);
        for (int64_t e = lo; e < hi; e++) {
            const JssHostInst &hi_ = a->insts[a->env_inst[e]];
            Cols c;
            const float d7[7] = {1.0f, (float)hi_.max_time_op, (float)hi_.M, (float)hi_.max_time_jobs,
                                 (float)hi_.max_time_op, (float)hi_.sum_op, (float)hi_.sum_op};
            for (int k = 0; k < 16; k++) { c.d[k] = k < 14 ? d7[k % 7] : 1.0f; c.r[k] = 1.0f / c.d[k]; }
            const uint8_t *row = a->wire + (size_t)e * a->wire_stride;
            const int t = a->scalars[4 * (size_t)e + 2];
            float *dst = a->obs + (size_t)e * a->jobs_max * 7;
            const size_t n = (size_t)hi_.J * 7;
#ifdef JSS_HAVE_AVX2_TARGET
            if (have_avx512() || have_avx2()) {
                if (have_avx512()) expand_env_avx512(row, hi_.J, hi_.M, t, hi_.len, c, stage.data());
                else expand_env_avx2(row, hi_.J, hi_.M, t, hi_.len, c, stage.data());
                stream_copy(dst, stage.data(), n);
                continue;
            }
#endif
            expand_env_scalar(row, hi_.J, hi_.M, t, hi_.len, c, dst);
        }
#ifdef JSS_HAVE_AVX2_TARGET
        if (have_avx2()) _mm_sfence();
#endif
    };
    Pool::get().parallel_for(a->env_end - a->env_begin, 256, [&](int64_t b, int64_t e) { work(a->env_begin + b, a->env_begin + e); });
}
