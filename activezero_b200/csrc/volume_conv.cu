// First 3-D convolution of the aggregation with the cost volume left IMPLICIT (SURVEY.md §8f rank 2, the
// "never materialise [B,64,Dq,Hq,Wq]" clause).
// Reference: /root/reference/nets/psmnet/psmnet.py:151-165 builds the concat volume, :165-168 feeds it to
// dres0 = convbn_3d(64, 32, 3, 1, 1) + ReLU + ...  (psmnet_submodule.py:44-56: Conv3d(bias=False) + BatchNorm3d).
//
//   out[b,co,d,y,x] = sum_{ci<64} sum_{kd,ky,kx<3} Wt[co,ci,kd,ky,kx] * vol[b,ci,d+kd-1,y+ky-1,x+kx-1]   (zero padding)
//   vol[b,ci,d',y',x']    = L[b,ci,y',x']        for x' >= d', else 0        (ci < 32)
//   vol[b,32+ci,d',y',x'] = R[b,ci,y',x'-d']     for x' >= d', else 0
//
// This is the one place on the hot path that is a dense contraction, so it runs on the 5th-generation tensor
// cores: an implicit GEMM with M = 128 consecutive x positions of one (b, d, y) row, N = 32 output channels and
// K = 27 taps x 64 channels, TF32 operands, fp32 accumulation in TENSOR MEMORY.
//   * the A operand is GATHERED straight from the two feature maps (left half: the row itself, masked below the
//     diagonal x' < d'; right half: the row shifted by d') into shared memory in the canonical K-major core-matrix
//     layout (8 rows x 16 bytes, no swizzle), rounded to TF32 (cvt.rna) -- one 130-row slab per (kd, ky), which the
//     three kx taps read through descriptors whose start address differs by one 16-byte row; the 401 MB-per-pair
//     volume and cuDNN's re-read of it disappear;
//   * the B operand of a tap (32 x 64 weights) is pre-packed on the device once per weight tensor in the same
//     core-matrix order and copied linearly;
//   * one elected thread issues 3 x 8 tcgen05.mma.cta_group::1.kind::tf32 (M128 N32 K8) per slab and commits them
//     to an mbarrier; two shared-memory stages, so the gather of slab t+1 overlaps the MMAs of slab t;
//   * epilogue: tcgen05.ld (32 lanes x 32 columns per warp) -> optional per-channel scale / shift (an eval-mode
//     BatchNorm folded in) and ReLU -> coalesced stores in NCDHW.
// grid = (ceil(W/128), H, Dq*B), 256 threads, 116 KB dynamic shared memory, 32 TMEM columns.
#include "common.cuh"

namespace az {

constexpr int kVcThreads = 256, kVcM = 128, kVcN = 32, kVcC = 32, kVcK = 64;
constexpr int kVcSlabGroups = 17;                        // 8-row groups of a slab: rows u = 0..135, 130 of them used
constexpr int kVcChunk = kVcSlabGroups * 8 * 16;         // bytes of one 4-channel chunk of a slab (rows at 16 B)
constexpr int kVcABytes = (kVcK / 4) * kVcChunk;         // 16 chunks = 64 channels
constexpr int kVcBBytes = 3 * kVcN * kVcK * 4;           // the three kx taps of a (kd, ky)
constexpr int kVcStage = kVcABytes + kVcBBytes;

__device__ __forceinline__ uint64_t vc_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    // cute::UMMA::SmemDescriptor: start address [0,14), leading byte offset [16,30), stride byte offset [32,46)
    // (all >> 4), version 1 at [46,48), base offset 0, layout type [61,64) = 0 (no swizzle)
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46);
}

// cute::UMMA::InstrDescriptor: c_format F32 (1) at [4,6), a/b format TF32 (2) at [7,10) / [10,13), both K-major,
// N >> 3 at [17,23), M >> 4 at [24,29)
constexpr uint32_t kVcIdesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(kVcN >> 3) << 17) | ((uint32_t)(kVcM >> 4) << 24);

__device__ __forceinline__ float to_tf32(float x) {
    uint32_t u;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
    return __uint_as_float(u);
}

// T = the features' and the output's element type: float, or bf16 / fp16 (widened at the gather, rounded once at the store)
template <typename T>
__global__ void __launch_bounds__(kVcThreads) volume_conv0_kernel(const T* __restrict__ L, const T* __restrict__ R,
                                                                  const float* __restrict__ wpacked,
                                                                  const float* __restrict__ scale,
                                                                  const float* __restrict__ shift, T* __restrict__ out,
                                                                  int B, int H, int W, int Dq, int relu) {
    extern __shared__ __align__(128) unsigned char vsm[];
    __shared__ __align__(8) uint64_t bars[2];
    __shared__ uint32_t tmem_base_s;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int x0 = blockIdx.x * kVcM, y = blockIdx.y;
    const int d = blockIdx.z % Dq, b = blockIdx.z / Dq;
    const size_t HW = (size_t)H * W;
    const uint32_t sbase = smem_u32(vsm);

    if (tid == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        mbar_fence_init();
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(32));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = tmem_base_s;

    const int r = lane & 7, e = lane >> 3;  // row within a core matrix, element within its 16-byte row
    int it = 0;                             // (kd, ky) slabs issued so far
    for (int kdy = 0; kdy < 9; ++kdy) {
        const int kd = kdy / 3, ky = kdy % 3;
        const int dp = d + kd - 1, yp = y + ky - 1;
        if (dp < 0 || dp >= Dq || yp < 0 || yp >= H) continue;  // these three taps read the volume's zero padding
        const int stage = it & 1;
        if (it >= 2) mbar_wait(&bars[stage], (uint32_t)(((it >> 1) - 1) & 1));  // the MMAs that read this stage are done
        unsigned char* As = vsm + (size_t)stage * kVcStage;
        unsigned char* Bs = As + kVcABytes;
        // ---- B: the three kx taps of (kd, ky) are consecutive in wpacked: 24 KB, linear copy
        {
            const float4* src = reinterpret_cast<const float4*>(wpacked + (size_t)(3 * kdy) * kVcN * kVcK);
            float4* dst = reinterpret_cast<float4*>(Bs);
#pragma unroll
            for (int k = 0; k < 6; ++k) dst[tid + k * kVcThreads] = __ldg(src + tid + k * kVcThreads);
        }
        // ---- A: ONE slab per (kd, ky) serves the three kx taps.  In the no-swizzle K-major layout a 4-channel chunk
        //      is linear in the row: byte 16 m + 4 e (8 rows x 16 B per core matrix, SBO = 128 B), so tap kx is the same
        //      slab read from a start address kx * 16 bytes further.  Slab row u holds volume column x' = x0 + u - 1.
        //      Warp w gathers the chunks kq = 2w, 2w+1 (k = 4 kq + e) for the 17 row groups; all of a thread's loads
        //      are issued before the first one is consumed (the gather is latency-bound).
        {
            float v[2][kVcSlabGroups];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int ci = 4 * (2 * warp + h) + e;
                const bool right = ci >= kVcC;
                const T* plane = (right ? R : L) + ((size_t)b * kVcC + (right ? ci - kVcC : ci)) * HW + (size_t)yp * W;
                const int sh = right ? dp : 0;
#pragma unroll
                for (int ug = 0; ug < kVcSlabGroups; ++ug) {
                    const int xp = x0 + 8 * ug + r - 1;
                    v[h][ug] = (xp >= dp && xp < W && xp >= 0) ? ld_f32(plane + xp - sh) : 0.f;
                }
            }
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                unsigned char* dstk = As + (size_t)(2 * warp + h) * kVcChunk + (size_t)r * 16 + (size_t)e * 4;
#pragma unroll
                for (int ug = 0; ug < kVcSlabGroups; ++ug) *reinterpret_cast<float*>(dstk + (size_t)ug * 128) = to_tf32(v[h][ug]);
            }
        }
        fence_async_smem();  // generic-proxy writes -> visible to the tensor core's async proxy
        __syncthreads();
        if (tid == 0) {
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t a0 = sbase + (uint32_t)stage * kVcStage, b0 = a0 + kVcABytes;
#pragma unroll
            for (int kx = 0; kx < 3; ++kx) {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    // K8 slice j = chunks 2j and 2j+1 (LBO = chunk stride), rows linear at 16 B (SBO = 128 B per 8 rows)
                    const uint64_t da = vc_smem_desc(a0 + (uint32_t)(2 * j) * kVcChunk + (uint32_t)kx * 16, kVcChunk, 128);
                    const uint64_t db = vc_smem_desc(b0 + (uint32_t)kx * (kVcN * kVcK * 4) + j * 1024, 512, 128);
                    const uint32_t acc = (it > 0 || kx > 0 || j > 0) ? 1u : 0u;
                    asm volatile(
                        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, {%5, %6, %7, %8}, p;\n\t}"
                        ::"r"(tmem), "l"(da), "l"(db), "r"(kVcIdesc), "r"(acc), "r"(0), "r"(0), "r"(0), "r"(0)
                        : "memory");
                }
            }
            // completion of everything issued so far -> this stage's barrier (implies fence::before_thread_sync)
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(&bars[stage]))
                         : "memory");
        }
        ++it;
    }
    // all MMAs complete in order: the last commit covers them
    {
        const int last = it - 1;
        mbar_wait(&bars[last & 1], (uint32_t)((last >> 1) & 1));
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    }
    if (warp < 4) {
        uint32_t v[32];
        const uint32_t taddr = tmem + ((uint32_t)(32 * warp) << 16);
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
            "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
            "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
            : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
              "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
              "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
              "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
            : "r"(taddr));
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        const int x = x0 + 32 * warp + lane;
        if (x < W) {
            T* o = out + (((size_t)b * kVcN) * Dq + d) * HW + (size_t)y * W + x;
            const size_t cstride = (size_t)Dq * HW;
#pragma unroll
            for (int n = 0; n < kVcN; ++n) {
                float val = __uint_as_float(v[n]);
                if (scale != nullptr) val = fmaf(val, __ldg(scale + n), __ldg(shift + n));
                if (relu) val = fmaxf(val, 0.f);
                st_from_f32(o + (size_t)n * cstride, val);
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(32));
}

// Packs a Conv3d weight [32][64][3][3][3] into the per-tap core-matrix order the kernel copies into shared memory:
// wpacked[tap][j = k/8][kc = (k/4)&1][ng = n/8][r = n%8][e = k%4], rounded to TF32.  grid = 27, 256 threads.
// DT = AZ_DTYPE_BF16 / AZ_DTYPE_F16 rounds each weight to that dtype first (RNE; what torch.autocast does to the weight
// of a cuDNN convolution), which TF32 then holds exactly; DT = 0 rounds to TF32 only.
template <int DT>
__global__ void __launch_bounds__(256) volume_conv0_pack_kernel(const float* __restrict__ w, float* __restrict__ wpacked) {
    const int tap = blockIdx.x;
    for (int t = threadIdx.x; t < kVcN * kVcK; t += 256) {
        const int e = t & 3, r = (t >> 2) & 7, ng = (t >> 5) & 3, kc = (t >> 7) & 1, j = t >> 8;
        const int n = 8 * ng + r, k = 8 * j + 4 * kc + e;
        float v = __ldg(w + ((size_t)n * kVcK + k) * 27 + tap);
        if (DT == AZ_DTYPE_BF16) v = __bfloat162float(__float2bfloat16_rn(v));
        if (DT == AZ_DTYPE_F16) v = __half2float(__float2half_rn(v));
        v = to_tf32(v);
        wpacked[(size_t)tap * kVcN * kVcK + t] = v;
        // second copy of the LEFT half (k < 32) in the N = 96 operand order of volume_conv_v2.cu, after the 27 tap
        // blocks: [kd*3+ky][j][kc][kx][ng][r][e] -- 12 KB per (kd, ky), one bulk copy each
        if (k < 32) {
            const int kdky = tap / 3, kx = tap - 3 * kdky;
            wpacked[(size_t)27 * kVcN * kVcK + (size_t)kdky * 3072 + j * 768 + kc * 384 + kx * 128 + ng * 32 + r * 4 + e] = v;
        }
    }
}

// volume_conv_v2.cu: shifted-coordinate, feature-stationary form (default when Dq <= 55)
template <typename T>
int volume_conv0_v2_launch(const T* L, const T* R, const float* wpacked, const float* scale, const float* shift,
                           T* out, int B, int H, int W, int Dq, int relu, cudaStream_t st, bool* done);

template <typename T>
int volume_conv0_fwd_launch(const T* L, const T* R, const float* wpacked, const float* scale, const float* shift, T* out,
                            int64_t B, int64_t H, int64_t W, int64_t Dq, int relu, cudaStream_t st) {
    if (tuning("AZ_VCONV", 2) == 2) {
        bool done = false;
        const int rc = volume_conv0_v2_launch<T>(L, R, wpacked, scale, shift, out, (int)B, (int)H, (int)W, (int)Dq, relu,
                                                 st, &done);
        if (rc != 0) return rc;
        if (done) return 0;
    }
    const size_t smem = 2 * (size_t)kVcStage;
    cudaError_t e = cudaFuncSetAttribute(volume_conv0_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    dim3 grid((unsigned)ceil_div(W, kVcM), (unsigned)H, (unsigned)(Dq * B));
    volume_conv0_kernel<T><<<grid, kVcThreads, smem, st>>>(L, R, wpacked, scale, shift, out, (int)B, (int)H, (int)W, (int)Dq,
                                                         relu);
    AZ_LAUNCH_CHECK();
    return 0;
}

}  // namespace az

using namespace az;

extern "C" int az_volume_conv0_pack(const float* weight, float* wpacked, void* stream) {
    if (!weight || !wpacked) return AZ_ERR_BAD_ARG;
    volume_conv0_pack_kernel<0><<<27, 256, 0, (cudaStream_t)stream>>>(weight, wpacked);
    AZ_LAUNCH_CHECK();
    return 0;
}

extern "C" int az_volume_conv0_pack_16(const float* weight, float* wpacked, int dtype, void* stream) {
    if (!weight || !wpacked || (dtype != AZ_DTYPE_BF16 && dtype != AZ_DTYPE_F16)) return AZ_ERR_BAD_ARG;
    if (dtype == AZ_DTYPE_BF16) volume_conv0_pack_kernel<AZ_DTYPE_BF16><<<27, 256, 0, (cudaStream_t)stream>>>(weight, wpacked);
    else volume_conv0_pack_kernel<AZ_DTYPE_F16><<<27, 256, 0, (cudaStream_t)stream>>>(weight, wpacked);
    AZ_LAUNCH_CHECK();
    return 0;
}

static int volume_conv0_check(const void* L, const void* R, const float* wpacked, const float* scale, const float* shift,
                              const void* out, int64_t B, int64_t C, int64_t H, int64_t W, int64_t Dq) {
    if (!L || !R || !wpacked || !out || B <= 0 || H <= 0 || W <= 0 || Dq <= 0) return AZ_ERR_BAD_ARG;
    if (C != kVcC || (scale == nullptr) != (shift == nullptr)) return AZ_ERR_BAD_ARG;  // PSMNet: 32 + 32 -> 32 channels
    if (H > 65535 || Dq * B > 65535 || H * W >= (1ll << 31) || !aligned16(wpacked)) return AZ_ERR_BAD_ARG;
    return 0;
}

extern "C" int az_volume_conv0_fwd(const float* L, const float* R, const float* wpacked, const float* scale,
                                   const float* shift, float* out, int64_t B, int64_t C, int64_t H, int64_t W,
                                   int64_t Dq, int relu, void* stream) {
    const int rc = volume_conv0_check(L, R, wpacked, scale, shift, out, B, C, H, W, Dq);
    if (rc != 0) return rc;
    return volume_conv0_fwd_launch<float>(L, R, wpacked, scale, shift, out, B, H, W, Dq, relu, (cudaStream_t)stream);
}

extern "C" int az_volume_conv0_fwd_16(const void* L, const void* R, const float* wpacked, const float* scale,
                                      const float* shift, void* out, int64_t B, int64_t C, int64_t H, int64_t W,
                                      int64_t Dq, int relu, int dtype, void* stream) {
    const int rc = volume_conv0_check(L, R, wpacked, scale, shift, out, B, C, H, W, Dq);
    if (rc != 0) return rc;
    if (dtype == AZ_DTYPE_BF16)
        return volume_conv0_fwd_launch<__nv_bfloat16>(static_cast<const __nv_bfloat16*>(L), static_cast<const __nv_bfloat16*>(R),
                                                      wpacked, scale, shift, static_cast<__nv_bfloat16*>(out), B, H, W, Dq,
                                                      relu, (cudaStream_t)stream);
    if (dtype == AZ_DTYPE_F16)
        return volume_conv0_fwd_launch<__half>(static_cast<const __half*>(L), static_cast<const __half*>(R), wpacked, scale,
                                               shift, static_cast<__half*>(out), B, H, W, Dq, relu, (cudaStream_t)stream);
    return AZ_ERR_BAD_ARG;
}
