// Host worker pool (jssenv_b200/csrc/jss_host.cpp): jss_host_parallel_for must return only once every chunk is done,
// also in the first regions after jss_host_pool_configure() restarted the workers (bench.py's e2e calibration does
// that between regions).  usage: check_pool iterations   (prints "<k> early returns"; exit status 1 if k > 0)
#include <atomic>
#include <cstdio>
#include <cstdlib>

#include "jss_host.h"

static std::atomic<long> g_done{0};

static void chunk(int64_t b, int64_t e, void *) {
    for (int64_t i = b; i < e; i++) {
        volatile double x = 0;
        for (int k = 0; k < 200; k++) x += k;
        g_done++;
    }
}

int main(int argc, char **argv) {
    const int iterations = argc > 1 ? atoi(argv[1]) : 1000;
    const int64_t n = 4096;
    int early = 0;
    for (int it = 0; it < iterations; it++) {
        jss_host_pool_configure(8, nullptr, 0);      // 7 workers + the caller, whatever the host has
        for (int r = 0; r < 2; r++) {
            g_done = 0;
            jss_host_parallel_for(n, 16, chunk, nullptr);
            if (g_done.load() != n) early++;
        }
    }
    printf("%d iterations, %d early returns\n", iterations, early);
    return early != 0;
}
