// Shared device/host helpers for libaz_stereo (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "../../include/az_stereo.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libaz_stereo is written for sm_100a (B200) only"
#endif

#define AZ_LAUNCH_CHECK() \
    do { cudaError_t e__ = cudaGetLastError(); if (e__ != cudaSuccess) return (int)e__; } while (0)

namespace az {

constexpr int kNumSMs = 148;  // B200: 2 dies x 74 SMs

// Developer knob: integer environment variable read at every call (kernel-variant A/B runs in
// benchmarks/variant_bench.py); absent => `dflt`.  Not part of the ABI contract.
inline int tuning(const char* name, int dflt) {
    const char* v = getenv(name);
    return (v && *v) ? atoi(v) : dflt;
}

__host__ __device__ inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// ---- streaming (evict-first) 128-bit / 32-bit global accesses ---------------------------
// The volumes (0.4-3.2 GB) are far larger than the 126 MB L2 and are consumed by a later
// kernel (cuDNN), so they are written/read with the .cs policy to keep L2 for the small inputs.
__device__ __forceinline__ void st_stream(float4* p, const float4& v) { __stcs(p, v); }
__device__ __forceinline__ void st_stream(float* p, float v) { __stcs(p, v); }
__device__ __forceinline__ float4 ld_stream(const float4* p) { return __ldcs(p); }
__device__ __forceinline__ float ld_stream(const float* p) { return __ldcs(p); }

// ---- 256-bit global accesses (sm_100: LDG.E.256 / STG.E.256; 32-byte aligned addresses) ----------------
struct __align__(32) float8 { float v[8]; };
inline bool aligned32(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 31u) == 0; }
__device__ __forceinline__ float8 ldg8(const float* p) {  // read-only path, like __ldg
    float8 r;
    asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(r.v[0]), "=f"(r.v[1]), "=f"(r.v[2]), "=f"(r.v[3]), "=f"(r.v[4]), "=f"(r.v[5]), "=f"(r.v[6]), "=f"(r.v[7])
                 : "l"(p));
    return r;
}
__device__ __forceinline__ void st_stream8(float* p, const float8& r) {  // evict-first, like __stcs
    asm volatile("st.global.cs.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "f"(r.v[0]), "f"(r.v[1]), "f"(r.v[2]),
                 "f"(r.v[3]), "f"(r.v[4]), "f"(r.v[5]), "f"(r.v[6]), "f"(r.v[7])
                 : "memory");
}

// ---- fp32 / 16-bit element access for kernels templated on the tensor dtype ----------------------------
// ld_f32: load one element and widen it to fp32 (exact for bf16 and fp16); st_from_f32: round once to the element
// type, to nearest even, and store.
__device__ __forceinline__ float ld_f32(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ld_f32(const __nv_bfloat16* p) { return __bfloat162float(__ldg(p)); }
__device__ __forceinline__ float ld_f32(const __half* p) { return __half2float(__ldg(p)); }
__device__ __forceinline__ void st_from_f32(float* p, float v) { *p = v; }
__device__ __forceinline__ void st_from_f32(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
__device__ __forceinline__ void st_from_f32(__half* p, float v) { *p = __float2half_rn(v); }

// ---- block reductions ---------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
// Sum over the CTA; result valid in thread 0.  `scratch` holds >= 32 doubles.
__device__ __forceinline__ double block_sum(double v, double* scratch) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) scratch[wid] = v;
    __syncthreads();
    double r = 0.0;
    if (wid == 0) {
        r = lane < nw ? scratch[lane] : 0.0;
        r = warp_sum(r);
    }
    return r;
}


// ---- mbarrier + 1-D bulk async copy (TMA, cp.async.bulk -> SASS UBLKCP) -------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// global -> shared, `bytes` a multiple of 16, both addresses 16-byte aligned; completes on `bar`
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// shared -> global (bulk group completion)
__device__ __forceinline__ void bulk_s2g(void* dst_gmem, const void* src_smem, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_u32(src_smem)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait() { asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory"); }
// make generic-proxy writes to shared memory visible to the async proxy (before a bulk store reads them)
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// 2^x with the MUFU unit only (2 ulp, denormal results flushed to zero).  exp2f() wraps the same
// instruction in a range fix-up for x < -126 (3 extra instructions per call) that softmax terms
// below 2^-126 of the maximum do not need.
__device__ __forceinline__ float fast_ex2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// ---- sample position of apply_disparity, in the reference's fp32 op order -----------------
// utils/reprojection.py:15-32 + grid_sample's unnormalise (align_corners=False):
//   f = lin[j] + disp/W;  g = 2*f - 1;  xs = ((g + 1) * W - 1) / 2
// torch's CPU grid_sampler fuses the (g+1)*W-1 step into one FMA (verified bit-for-bit against
// F.grid_sample in the authoring container), so the same contraction is spelled out here and
// everything else is kept un-fused with the _rn intrinsics.
__device__ __forceinline__ float sample_pos(float lin, float shift, float size) {
    const float f = __fadd_rn(lin, shift);
    const float g = __fsub_rn(__fmul_rn(2.0f, f), 1.0f);
    return __fmul_rn(__fmaf_rn(__fadd_rn(g, 1.0f), size, -1.0f), 0.5f);
}

// ---- one axis of a bilinear sample: cell index, weights and zero-padding validity ----------
struct Axis {
    int i0;      // floor(pos), clamped to [-2, size] so it is safe to form indices from
    float w, e;  // w = pos - floor(pos), e = 1 - w
    bool v0, v1; // corner i0 / i0+1 inside [0,size)
};

__device__ __forceinline__ Axis make_axis(float pos, int size) {
    Axis a;
    const float fl = floorf(pos);
    a.w = __fsub_rn(pos, fl);
    a.e = __fsub_rn(1.0f, a.w);
    a.v0 = (fl >= 0.0f) && (fl <= (float)(size - 1));
    a.v1 = (fl >= -1.0f) && (fl <= (float)(size - 2));
    a.i0 = (int)fminf(fmaxf(fl, -2.0f), (float)size);
    return a;
}

}  // namespace az
