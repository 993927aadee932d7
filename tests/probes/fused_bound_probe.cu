// Evaluates the fused-classification helpers of the RANSAC scoring kernels (evenvizion_b200/csrc/ransac_device.cuh)
// exactly as the kernels compile them, one (f32 model, point pair, t, cmax) per element, so that tests can compare them
// with the NumPy restatements in oracle/ransac.py.  All pointers are device pointers (torch tensors); nothing is copied.
#include "ransac_device.cuh"

namespace {

__global__ void fused_bound_probe_kernel(const float* __restrict__ h, const float4* __restrict__ p, const float* __restrict__ t,
                                         const float* __restrict__ cmax, int64_t n, float* e_fused, float* e_exact,
                                         float* tlo, float* thi, uint8_t* safe, float* rcp, float* den_f, float* den_e) {
    for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n;
         i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        float hf[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) hf[k] = h[i * 8 + k];
        const float4 pt = p[i];
        e_fused[i] = evz::reproj_err_fused(hf, pt);
        e_exact[i] = evz::reproj_err32(hf, pt);
        evz::FhArgs a{};
        a.thresh2 = t[i];
        evz::set_fused_cut(a);
        float lo, hi;
        evz::fused_thresholds(hf, cmax[i], a, false, lo, hi);
        tlo[i] = lo;
        thi[i] = hi;
        safe[i] = evz::den_safe(hf[6], hf[7], cmax[i]) ? 1 : 0;
        // the denominators of both paths, and the reciprocal reproj_err_fused uses
        const float df = __fmaf_rn(hf[6], pt.x, __fmaf_rn(hf[7], pt.y, 1.f));
        float ww;
        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(ww) : "f"(df));
        den_f[i] = df;
        rcp[i] = ww;
        den_e[i] = __fadd_rn(__fadd_rn(__fmul_rn(hf[6], pt.x), __fmul_rn(hf[7], pt.y)), 1.f);
    }
}

}  // namespace

// Returns 0, or the CUDA error of the launch.
extern "C" int fused_bound_probe(const float* h, const float* pts, const float* t, const float* cmax, int64_t n,
                                 float* e_fused, float* e_exact, float* tlo, float* thi, uint8_t* safe, float* rcp,
                                 float* den_f, float* den_e, cudaStream_t stream) {
    if (n <= 0) return 0;
    const int64_t blocks = (n + 255) / 256;
    fused_bound_probe_kernel<<<static_cast<unsigned>(blocks < 8192 ? blocks : 8192), 256, 0, stream>>>(
        h, reinterpret_cast<const float4*>(pts), t, cmax, n, e_fused, e_exact, tlo, thi, safe, rcp, den_f, den_e);
    return static_cast<int>(cudaGetLastError());
}
