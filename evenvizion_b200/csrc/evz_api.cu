// Handle lifetime, error text and scratch management of libevz.so.
#include "evz_common.cuh"

static char g_create_err[512] = "";

extern "C" int evz_version(void) { return EVZ_VERSION; }

extern "C" int evz_create(int device, evz_handle** out) {
    if (!out) return EVZ_E_ARG;
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) {
        snprintf(g_create_err, sizeof(g_create_err), "evz_create: no CUDA device (%s); this library has no CPU fallback",
                 e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
        return EVZ_E_NODEVICE;
    }
    if (device < 0 || device >= n) {
        snprintf(g_create_err, sizeof(g_create_err), "evz_create: device %d out of range [0,%d)", device, n);
        return EVZ_E_ARG;
    }
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) {
        snprintf(g_create_err, sizeof(g_create_err), "evz_create: %s", cudaGetErrorString(e));
        return EVZ_E_CUDA;
    }
    if (prop.major != 10) {
        snprintf(g_create_err, sizeof(g_create_err), "evz_create: device %d is sm_%d%d; libevz is built for sm_100a (B200) only",
                 device, prop.major, prop.minor);
        return EVZ_E_UNSUPPORTED;
    }
    e = cudaSetDevice(device);
    if (e != cudaSuccess) {
        snprintf(g_create_err, sizeof(g_create_err), "evz_create: cudaSetDevice: %s", cudaGetErrorString(e));
        return EVZ_E_CUDA;
    }
    evz_handle* h = new evz_handle();
    h->device = device;
    h->sm_count = prop.multiProcessorCount;
    *out = h;
    return EVZ_OK;
}

extern "C" void evz_destroy(evz_handle* h) {
    if (!h) return;
    if (h->scratch) cudaFree(h->scratch);
    if (h->match_ev_made)
        for (auto& pr : h->match_ev) { cudaEventDestroy(pr[0]); cudaEventDestroy(pr[1]); }
    delete h;
}

extern "C" const char* evz_last_error(const evz_handle* h) { return h ? h->err : g_create_err; }

extern "C" int evz_sm_count(const evz_handle* h) { return h ? h->sm_count : 0; }

extern "C" int evz_set_option(evz_handle* h, int option, int value) {
    if (!h) return EVZ_E_ARG;
    switch (option) {
        case EVZ_OPT_RANSAC_EXACT: h->opt_ransac_exact = value; return EVZ_OK;
        case EVZ_OPT_MATCH_VARIANT:
            EVZ_REQUIRE(h, value == 0 || value == 5, "EVZ_OPT_MATCH_VARIANT must be 0 (default routing) or 5 (key-space kernel for every pair)");
            h->opt_match_variant = value; return EVZ_OK;
        case EVZ_OPT_RANSAC_NO_PRUNE: h->opt_ransac_no_prune = value; return EVZ_OK;
        case EVZ_OPT_TIME_MATCH: h->opt_time_match = value; return EVZ_OK;
        default: EVZ_SET_ERR(h, "evz_set_option: unknown option %d", option); return EVZ_E_ARG;
    }
}

extern "C" int evz_match_kernel_ms(evz_handle* h, int k, float* ms) {
    if (!h || !ms) return EVZ_E_ARG;
    EVZ_REQUIRE(h, h->match_ev_made && k >= 0 && k < 16 && static_cast<unsigned long long>(k) < h->match_calls,
                "no timing record (set EVZ_OPT_TIME_MATCH and call evz_match_top2 first)");
    const auto& pr = h->match_ev[(h->match_calls - 1 - k) & 15];
    EVZ_CUDA_CHECK(h, cudaEventElapsedTime(ms, pr[0], pr[1]));
    return EVZ_OK;
}

int evz_scratch(evz_handle* h, size_t bytes, void** out) {
    if (bytes > h->scratch_bytes) {
        // growing is the one place the library synchronises: work queued on the old block must finish
        EVZ_CUDA_CHECK(h, cudaDeviceSynchronize());
        if (h->scratch) { cudaFree(h->scratch); h->scratch = nullptr; h->scratch_bytes = 0; }
        const size_t want = evz_align_up(bytes + bytes / 4, size_t(1) << 20);
        cudaError_t e = cudaMalloc(&h->scratch, want);
        if (e != cudaSuccess) {
            (void)cudaGetLastError();          // reported here, not again by the next launch check
            EVZ_SET_ERR(h, "scratch allocation of %zu bytes failed: %s", want, cudaGetErrorString(e));
            return EVZ_E_NOMEM;
        }
        h->scratch_bytes = want;
    }
    *out = h->scratch;
    return EVZ_OK;
}
