// Shared host-side plumbing of libevz.so: handle, error reporting, scratch.
#pragma once
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <cuda.h>
#include <cuda_runtime.h>
#include "../../include/evz.h"

typedef CUresult (*evz_encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                        const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                        CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                        CUtensorMapFloatOOBfill);

struct evz_handle {
    int device = 0;
    int sm_count = 0;
    char err[512] = {0};
    // grow-only scratch
    void* scratch = nullptr;
    size_t scratch_bytes = 0;
    // cached TMA descriptor of the descriptor store
    CUtensorMap tmap;
    const void* tmap_ptr = nullptr;
    int64_t tmap_rows = 0;
    evz_encode_tiled_fn encode = nullptr;
    // cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is per device: remembered per handle, not per process
    unsigned attr_match = 0;       // bit 0: key-space kernel, bit 1: V-space kernel
    bool attr_static = false, attr_canon = false, attr_concat = false;
    int attr_filter = 0, attr_score = 0, attr_score_g = 0, attr_score_a = 0, attr_refit = 0;
    int score_smem_room = -1;      // dynamic shared memory a scoring block may take (-1: not queried yet)
    // options (evz_set_option)
    int opt_ransac_exact = 0;
    int opt_ransac_no_prune = 0;
    int opt_match_variant = 0;
    int opt_time_match = 0;
    // EVZ_OPT_TIME_MATCH: ring of event pairs around the main match kernel
    cudaEvent_t match_ev[16][2] = {};
    bool match_ev_made = false;
    unsigned long long match_calls = 0;
};

#define EVZ_SET_ERR(h, ...) do { if (h) snprintf((h)->err, sizeof((h)->err), __VA_ARGS__); } while (0)

// A failure is reported once: the runtime's last-error state is cleared, so that the next cudaGetLastError() -- the
// launch check of a later call, or PyTorch's -- does not report it again against unrelated work.
#define EVZ_CUDA_CHECK(h, expr) do { cudaError_t e__ = (expr); if (e__ != cudaSuccess) {            \
        EVZ_SET_ERR(h, "%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(e__));        \
        (void)cudaGetLastError(); return EVZ_E_CUDA; } } while (0)

#define EVZ_LAUNCH_CHECK(h) EVZ_CUDA_CHECK(h, cudaGetLastError())

// every entry point runs on the handle's device, whatever device the calling thread had current
#define EVZ_ENTER(h) do { int d__ = -1; if (cudaGetDevice(&d__) != cudaSuccess || d__ != (h)->device)                     \
        EVZ_CUDA_CHECK(h, cudaSetDevice((h)->device)); } while (0)

#define EVZ_REQUIRE(h, cond, msg) do { if (!(cond)) { EVZ_SET_ERR(h, "%s: %s", __func__, msg); return EVZ_E_ARG; } } while (0)

// returns a device scratch region of at least `bytes` (256-byte aligned); contents undefined
int evz_scratch(evz_handle* h, size_t bytes, void** out);

static inline size_t evz_align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
