// Concat cost volume with 16-bit (bf16 / fp16) features, forward and backward: the volume torch.autocast's
// convolutions consume, written in their dtype (DESIGN.md §4.11).
//
// Forward: a copy of 2-byte elements, so one kernel per layout serves both dtypes.  The volume element is the
// feature element itself, i.e. exactly what the fp32 volume of the upcast features gives after .to(dtype).
// Backward: the fp32 kernels' sums (ascending i, one fp32 accumulator per output element, concat_volume.cu) of the
// upcast 16-bit gradient, rounded once to the feature dtype (RNE).  Adding +0 to an accumulator that started at +0
// never changes it, so the masked terms the vector loops add are harmless and the result equals the fp32 op on
// gvol.float() followed by .to(dtype), bit for bit.
#include "common.cuh"

namespace az {

constexpr int kF16DG = 8;  // disparity planes per forward thread (the octet window needs 8)

// 8 consecutive 2-byte elements = one 16-byte access
struct __align__(16) h8 { uint16_t v[8]; };
__device__ __forceinline__ h8 ldg_h8(const uint16_t* p) {
    const uint4 u = __ldg(reinterpret_cast<const uint4*>(p));
    h8 r;
    *reinterpret_cast<uint4*>(&r) = u;
    return r;
}
__device__ __forceinline__ void st_stream_h8(uint16_t* p, const h8& r) {
    __stcs(reinterpret_cast<uint4*>(p), *reinterpret_cast<const uint4*>(&r));
}
__device__ __forceinline__ h8 ld_stream_h8(const uint16_t* p) {
    const uint4 u = __ldcs(reinterpret_cast<const uint4*>(p));
    h8 r;
    *reinterpret_cast<uint4*>(&r) = u;
    return r;
}

template <int DT> __device__ __forceinline__ float h2f(uint16_t u);
template <> __device__ __forceinline__ float h2f<AZ_DTYPE_BF16>(uint16_t u) { return __uint_as_float((uint32_t)u << 16); }
template <> __device__ __forceinline__ float h2f<AZ_DTYPE_F16>(uint16_t u) { return __half2float(__ushort_as_half(u)); }
template <int DT> __device__ __forceinline__ uint16_t f2h(float x);
template <> __device__ __forceinline__ uint16_t f2h<AZ_DTYPE_BF16>(float x) { return __bfloat16_as_ushort(__float2bfloat16_rn(x)); }
template <> __device__ __forceinline__ uint16_t f2h<AZ_DTYPE_F16>(float x) { return __half_as_ushort(__float2half_rn(x)); }

// ------------------------------------------------------------------------------------------
// forward NCDHW, 16-byte accesses (W % 8 == 0, 16-byte aligned bases): concat_fwd_vec8_kernel with 2-byte elements.
// A thread owns 8 consecutive elements of one (b, channel) plane and writes them to the 8 planes i0 .. i0+7; the right
// half's shift by i = i0 + r is the window [8-r, 16-r) of two ALIGNED octets, A at x-i0-8 and B at x-i0
// (tests/test_concat_vec8_model.py models the index logic).  grid = (ceil(H*W/8 / 256), 2C * ceil(Dq/8), B).
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) concat16_fwd_vec8_kernel(const uint16_t* __restrict__ L, const uint16_t* __restrict__ R,
                                                                uint16_t* __restrict__ vol, int C, int H, int W, int Dq,
                                                                int ngroups) {
    const int W8 = W >> 3;
    const int oc = blockIdx.y / ngroups, dg = blockIdx.y - oc * ngroups, b = blockIdx.z;
    const int i0 = dg * kF16DG, i1 = min(Dq, i0 + kF16DG);
    const bool right = oc >= C;
    const int c = right ? oc - C : oc;
    const int p = blockIdx.x * 256 + threadIdx.x;
    if (p >= H * W8) return;
    const size_t HW = (size_t)H * W;
    const int x = (p % W8) * 8;
    const uint16_t* sp = (right ? R : L) + ((size_t)b * C + c) * HW + (size_t)p * 8;  // feature[y][x]
    uint16_t* op = vol + ((size_t)b * 2 * C + oc) * Dq * HW + (size_t)p * 8;
    if (!right) {
        const h8 v = ldg_h8(sp);
#pragma unroll
        for (int r = 0; r < kF16DG; ++r) {
            const int i = i0 + r;
            if (i >= i1) break;
            h8 o = v;
            if (x < i) {
#pragma unroll
                for (int k = 0; k < 8; ++k)
                    if (x + k < i) o.v[k] = 0;
            }
            st_stream_h8(op + (size_t)i * HW, o);
        }
    } else {
        uint16_t ab[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) ab[k] = 0;
        if (x - i0 >= 0) {
            const h8 Bv = ldg_h8(sp - i0);
#pragma unroll
            for (int k = 0; k < 8; ++k) ab[8 + k] = Bv.v[k];
        }
        if (x - i0 - 8 >= 0) {
            const h8 Av = ldg_h8(sp - i0 - 8);
#pragma unroll
            for (int k = 0; k < 8; ++k) ab[k] = Av.v[k];
        }
#pragma unroll
        for (int r = 0; r < kF16DG; ++r) {
            if (i0 + r >= i1) break;
            h8 o;
#pragma unroll
            for (int k = 0; k < 8; ++k) o.v[k] = ab[8 - r + k];
            st_stream_h8(op + (size_t)(i0 + r) * HW, o);
        }
    }
}

// forward NCDHW, scalar fallback (any W, any alignment): one thread per element of a (b, oc, i) plane.
// grid = (ceil(H*W/256), Dq, B*2C)
__global__ void __launch_bounds__(256) concat16_fwd_scalar_kernel(const uint16_t* __restrict__ L, const uint16_t* __restrict__ R,
                                                                  uint16_t* __restrict__ vol, int C, int H, int W, int Dq) {
    const int hw = blockIdx.x * 256 + threadIdx.x;
    if (hw >= H * W) return;
    const int i = blockIdx.y;
    const int boc = blockIdx.z, b = boc / (2 * C), oc = boc - b * 2 * C;
    const int x = hw % W;
    uint16_t v = 0;
    if (x >= i) {
        if (oc < C) v = L[((size_t)b * C + oc) * H * W + hw];
        else        v = R[((size_t)b * C + (oc - C)) * H * W + hw - i];
    }
    vol[(((size_t)boc * Dq + i) * H) * W + hw] = v;
}

// ------------------------------------------------------------------------------------------
// forward channels_last_3d (memory order [B][Dq][H][W][2C], C % 8 == 0): concat_fwd_ndhwc_kernel with 2-byte elements.
// A CTA owns 64 consecutive x of one (b, y) and kClDG planes; it stages the 64 left and 64 + 7 right feature vectors
// TRANSPOSED in shared memory (position-major, C elements per position, pitch C + 8), then writes every plane's
// 64 positions x 2C elements as one contiguous run of 16-byte streaming stores.  grid = (ntiles * ngroups, H, B).
// ------------------------------------------------------------------------------------------
constexpr int kCl16TX = 64, kCl16TXB = 32, kCl16DG = 8, kCl16Threads = 256;

__global__ void __launch_bounds__(kCl16Threads) concat16_fwd_ndhwc_kernel(const uint16_t* __restrict__ L,
                                                                        const uint16_t* __restrict__ R,
                                                                        uint16_t* __restrict__ vol, int C, int H, int W,
                                                                        int Dq, int ntiles) {
    extern __shared__ __align__(16) uint16_t hsm[];
    const int P = C + 8;  // pitch of one position (elements): a multiple of 8
    uint16_t* LsT = hsm;                // [kCl16TX][P]
    uint16_t* RsT = hsm + kCl16TX * P;  // [kCl16TX + kCl16DG - 1][P]: x0 - (i1-1) .. x0 + kCl16TX - 1
    const int tile = blockIdx.x % ntiles, dg = blockIdx.x / ntiles;
    const int i0 = dg * kCl16DG, i1 = min(Dq, i0 + kCl16DG);
    const int x0 = tile * kCl16TX, y = blockIdx.y, b = blockIdx.z;
    const int nr = kCl16TX + (i1 - i0) - 1;
    const size_t HW = (size_t)H * W;
    const uint16_t* Lb = L + (size_t)b * C * HW + (size_t)y * W;
    const uint16_t* Rb = R + (size_t)b * C * HW + (size_t)y * W;
    for (int t = threadIdx.x; t < C * kCl16TX; t += kCl16Threads) {
        const int c = t / kCl16TX, xl = t - c * kCl16TX, x = x0 + xl;
        LsT[xl * P + c] = x < W ? Lb[(size_t)c * HW + x] : (uint16_t)0;
    }
    for (int t = threadIdx.x; t < C * nr; t += kCl16Threads) {
        const int c = t / nr, r = t - c * nr, x = x0 - (i1 - 1) + r;
        RsT[r * P + c] = (x >= 0 && x < W) ? Rb[(size_t)c * HW + x] : (uint16_t)0;
    }
    __syncthreads();
    const int C8 = C >> 3, Q = 2 * C8;  // 16-byte vectors per position
    const int npos = min(kCl16TX, W - x0);
    const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
    uint16_t* vrow = vol + (((size_t)b * Dq * H + y) * W + x0) * (size_t)(2 * C);  // d = 0
    const size_t dstep = (size_t)H * W * (2 * C);
    if (Q <= kCl16Threads && (kCl16Threads % Q) == 0 && kCl16TX * Q <= 4 * kCl16Threads &&
        ((kCl16Threads / Q) >= kCl16TX || (kCl16TX % (kCl16Threads / Q)) == 0)) {
        // fast path (C = 8, 16, 32, 64, 128): a thread keeps its channel octet q and walks <= 4 positions
        const int q = threadIdx.x % Q, xstep = kCl16Threads / Q, nk = xstep >= kCl16TX ? 1 : kCl16TX / xstep;
        const bool left = q < C8;
        uint4 vl[4];
        const uint16_t* rp[4];
        int xs[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int xl = threadIdx.x / Q + k * xstep;
            xs[k] = (k < nk && xl < npos) ? x0 + xl : -1;  // -1: nothing to write
            vl[k] = zero;
            rp[k] = RsT;
            if (xs[k] >= 0) {
                if (left) vl[k] = *reinterpret_cast<const uint4*>(LsT + xl * P + 8 * q);
                else rp[k] = RsT + (xl + i1 - 1) * P + 8 * (q - C8);
            }
        }
        for (int d = i0; d < i1; ++d) {
            uint4* od = reinterpret_cast<uint4*>(vrow + (size_t)d * dstep) + threadIdx.x;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (xs[k] >= 0) {
                    uint4 v = zero;
                    if (xs[k] >= d) v = left ? vl[k] : *reinterpret_cast<const uint4*>(rp[k] - d * P);
                    __stcs(od + k * kCl16Threads, v);
                }
            }
        }
        return;
    }
    for (int d = i0; d < i1; ++d) {
        uint4* od = reinterpret_cast<uint4*>(vrow + (size_t)d * dstep);
        for (int t = threadIdx.x; t < npos * Q; t += kCl16Threads) {
            const int xl = t / Q, q = t - xl * Q;
            uint4 v = zero;
            if (x0 + xl >= d)
                v = q < C8 ? *reinterpret_cast<const uint4*>(LsT + xl * P + 8 * q)
                           : *reinterpret_cast<const uint4*>(RsT + (xl - d + i1 - 1) * P + 8 * (q - C8));
            __stcs(od + t, v);
        }
    }
}

// ------------------------------------------------------------------------------------------
// backward NCDHW, 16-byte loads (W % 8 == 0, aligned): concat_bwd_direct_kernel with octets.  One thread per 8
// elements of gL / gR, fp32 accumulators, ascending i.  Right half: output columns x..x+7 need g[i][x+i .. x+i+7];
// with i = 8m + r that is the window [r, r+8) of the two ALIGNED octets at columns x+8m and x+8m+8 (the second is
// zero when it lies right of the row).  grid = (ceil(H*W/8/256), 2C, B)
// ------------------------------------------------------------------------------------------
template <int DT>
__global__ void __launch_bounds__(256) concat16_bwd_vec8_kernel(const uint16_t* __restrict__ gvol, uint16_t* __restrict__ gL,
                                                                uint16_t* __restrict__ gR, int C, int H, int W, int Dq) {
    const int W8 = W >> 3;
    const int p = blockIdx.x * 256 + threadIdx.x;
    if (p >= H * W8) return;
    const int oc = blockIdx.y, b = blockIdx.z;
    const bool right = oc >= C;
    uint16_t* gout = right ? gR : gL;
    if (gout == nullptr) return;
    const int c = right ? oc - C : oc;
    const int x = (p % W8) * 8;
    const size_t HW = (size_t)H * W;
    const uint16_t* g = gvol + ((size_t)b * 2 * C + oc) * Dq * HW + (size_t)p * 8;
    float acc[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[k] = 0.f;
    if (!right) {
        const int lim = min(Dq, x + 8);  // planes i > x+7 only hold the zero triangle for these columns
        for (int i0 = 0; i0 < lim; i0 += 8) {
            h8 v[8];
#pragma unroll
            for (int r = 0; r < 8; ++r) {
                if (i0 + r < lim) v[r] = ld_stream_h8(g + (size_t)(i0 + r) * HW);
                else *reinterpret_cast<uint4*>(&v[r]) = make_uint4(0u, 0u, 0u, 0u);
            }
#pragma unroll
            for (int r = 0; r < 8; ++r) {
                const int i = i0 + r;
#pragma unroll
                for (int k = 0; k < 8; ++k) acc[k] += (x + k >= i) ? h2f<DT>(v[r].v[k]) : 0.f;
            }
        }
    } else {
        const int lim = min(Dq, W - x);  // x+i < W
        for (int m8 = 0; m8 < lim; m8 += 8) {
            h8 A[8], Bv[8];
            const bool inB = (x + m8 + 8) < W;
#pragma unroll
            for (int r = 0; r < 8; ++r) {
                const bool on = (m8 + r) < lim;
                const uint16_t* q = g + (size_t)(m8 + r) * HW + m8;
                *reinterpret_cast<uint4*>(&A[r]) = make_uint4(0u, 0u, 0u, 0u);
                *reinterpret_cast<uint4*>(&Bv[r]) = make_uint4(0u, 0u, 0u, 0u);
                if (on) A[r] = ldg_h8(q);
                if (on && inB) Bv[r] = ldg_h8(q + 8);
            }
#pragma unroll
            for (int r = 0; r < 8; ++r) {
#pragma unroll
                for (int k = 0; k < 8; ++k) acc[k] += h2f<DT>(r + k < 8 ? A[r].v[r + k] : Bv[r].v[r + k - 8]);
            }
        }
    }
    h8 o;
#pragma unroll
    for (int k = 0; k < 8; ++k) o.v[k] = f2h<DT>(acc[k]);
    *reinterpret_cast<uint4*>(gout + ((size_t)b * C + c) * HW + (size_t)p * 8) = *reinterpret_cast<const uint4*>(&o);
}

// backward NCDHW, scalar fallback: one thread per output element.  grid = (ceil(H*W/256), 2C, B)
template <int DT>
__global__ void __launch_bounds__(256) concat16_bwd_scalar_kernel(const uint16_t* __restrict__ gvol, uint16_t* __restrict__ gL,
                                                                  uint16_t* __restrict__ gR, int C, int H, int W, int Dq) {
    const int hw = blockIdx.x * 256 + threadIdx.x;
    if (hw >= H * W) return;
    const int oc = blockIdx.y, b = blockIdx.z;
    const bool right = oc >= C;
    uint16_t* gout = right ? gR : gL;
    if (gout == nullptr) return;
    const int c = right ? oc - C : oc;
    const int x = hw % W;
    const size_t HW = (size_t)H * W;
    const uint16_t* g = gvol + ((size_t)b * 2 * C + oc) * Dq * HW + hw;
    float acc = 0.f;
    if (right) {
        const int lim = min(Dq, W - x);
        for (int i = 0; i < lim; ++i) acc += h2f<DT>(g[(size_t)i * HW + i]);
    } else {
        const int lim = min(Dq, x + 1);
        for (int i = 0; i < lim; ++i) acc += h2f<DT>(g[(size_t)i * HW]);
    }
    gout[((size_t)b * C + c) * HW + hw] = f2h<DT>(acc);
}

// backward channels_last_3d (C % 8 == 0): concat_bwd_ndhwc_kernel with octets.  A 32-position tile; a thread owns
// (position, eight channels) and walks the Dq planes in ascending order (left: straight down; right: along x + d);
// the rounded sums are transposed through shared memory so that gL / gR are written as coalesced rows.
template <int DT>
__global__ void __launch_bounds__(kCl16Threads) concat16_bwd_ndhwc_kernel(const uint16_t* __restrict__ gvol,
                                                                        uint16_t* __restrict__ gL, uint16_t* __restrict__ gR,
                                                                        int C, int H, int W, int Dq) {
    extern __shared__ __align__(16) uint16_t hsm[];  // Ts[2C][kCl16TXB + 2]
    constexpr int TP = kCl16TXB + 2;
    const int x0 = blockIdx.x * kCl16TXB, y = blockIdx.y, b = blockIdx.z;
    const int C8 = C >> 3, Q = 2 * C8, C2 = 2 * C;
    const size_t plane = (size_t)H * W * C2;  // elements between consecutive disparities
    const uint16_t* gb = gvol + ((size_t)b * Dq * H + y) * (size_t)W * C2;
    for (int t = threadIdx.x; t < kCl16TXB * Q; t += kCl16Threads) {
        const int xl = t / Q, q = t - xl * Q, x = x0 + xl;
        const bool right = q >= C8;
        float acc[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) acc[k] = 0.f;
        if (x < W && (right ? gR != nullptr : gL != nullptr)) {
            // left: g[d][x] for d <= x;  right: g[d][x + d] while x + d < W
            const int nd = right ? min(Dq, W - x) : min(Dq, x + 1);
            const uint16_t* p = gb + (size_t)x * C2 + 8 * q;
            const size_t step = plane + (right ? (size_t)C2 : 0);
            int d = 0;
            for (; d + 8 <= nd; d += 8) {
                h8 v[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) v[k] = ld_stream_h8(p + (size_t)(d + k) * step);
#pragma unroll
                for (int k = 0; k < 8; ++k) {
#pragma unroll
                    for (int e = 0; e < 8; ++e) acc[e] += h2f<DT>(v[k].v[e]);
                }
            }
            for (; d < nd; ++d) {
                const h8 v = ld_stream_h8(p + (size_t)d * step);
#pragma unroll
                for (int e = 0; e < 8; ++e) acc[e] += h2f<DT>(v.v[e]);
            }
        }
        uint16_t* ts = hsm + (8 * q) * TP + xl;
#pragma unroll
        for (int e = 0; e < 8; ++e) ts[e * TP] = f2h<DT>(acc[e]);
    }
    __syncthreads();
    const size_t HW = (size_t)H * W;
    for (int t = threadIdx.x; t < C2 * kCl16TXB; t += kCl16Threads) {
        const int ch = t / kCl16TXB, xl = t - ch * kCl16TXB, x = x0 + xl;
        if (x >= W) continue;
        uint16_t* dst = ch < C ? gL : gR;
        if (dst == nullptr) continue;
        const int c = ch < C ? ch : ch - C;
        dst[((size_t)b * C + c) * HW + (size_t)y * W + x] = hsm[ch * TP + xl];
    }
}

template <int DT>
int concat16_bwd_launch(const uint16_t* g, uint16_t* gL, uint16_t* gR, int64_t B, int64_t C, int64_t H, int64_t W,
                        int64_t Dq, bool ndhwc, cudaStream_t st) {
    if (ndhwc) {
        const size_t smem = (size_t)(2 * C) * (kCl16TXB + 2) * sizeof(uint16_t);
        cudaError_t e = cudaFuncSetAttribute(concat16_bwd_ndhwc_kernel<DT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e != cudaSuccess) return (int)e;
        dim3 grid((unsigned)ceil_div(W, kCl16TXB), (unsigned)H, (unsigned)B);
        concat16_bwd_ndhwc_kernel<DT><<<grid, kCl16Threads, smem, st>>>(g, gL, gR, (int)C, (int)H, (int)W, (int)Dq);
        AZ_LAUNCH_CHECK();
        return 0;
    }
    const bool vec = (W % 8 == 0) && aligned16(g) && (!gL || aligned16(gL)) && (!gR || aligned16(gR));
    if (vec) {
        dim3 grid((unsigned)ceil_div(H * (W / 8), 256), (unsigned)(2 * C), (unsigned)B);
        concat16_bwd_vec8_kernel<DT><<<grid, 256, 0, st>>>(g, gL, gR, (int)C, (int)H, (int)W, (int)Dq);
        AZ_LAUNCH_CHECK();
        return 0;
    }
    dim3 grid((unsigned)ceil_div(H * W, 256), (unsigned)(2 * C), (unsigned)B);
    concat16_bwd_scalar_kernel<DT><<<grid, 256, 0, st>>>(g, gL, gR, (int)C, (int)H, (int)W, (int)Dq);
    AZ_LAUNCH_CHECK();
    return 0;
}

}  // namespace az

using namespace az;

extern "C" int az_concat_volume_fwd_16(const void* L, const void* R, void* vol, int64_t B, int64_t C, int64_t H, int64_t W,
                                       int64_t Dq, int channels_last, void* stream) {
    if (!L || !R || !vol || B <= 0 || C <= 0 || H <= 0 || W <= 0 || Dq <= 0) return AZ_ERR_BAD_ARG;
    if (H * W >= (1ll << 31) / 8 || B > 65535) return AZ_ERR_BAD_ARG;
    const uint16_t* l = static_cast<const uint16_t*>(L);
    const uint16_t* r = static_cast<const uint16_t*>(R);
    uint16_t* v = static_cast<uint16_t*>(vol);
    cudaStream_t st = (cudaStream_t)stream;
    if (channels_last) {
        if ((C % 8) != 0 || !aligned16(vol) || H > 65535) return AZ_ERR_BAD_ARG;
        const size_t smem = (size_t)(2 * kCl16TX + kCl16DG - 1) * (size_t)(C + 8) * sizeof(uint16_t);
        if (smem > 200 * 1024) return AZ_ERR_BAD_ARG;
        const int64_t ntiles = ceil_div(W, kCl16TX), ngroups = ceil_div(Dq, kCl16DG);
        if (ntiles * ngroups >= (1ll << 31)) return AZ_ERR_BAD_ARG;
        cudaError_t e = cudaFuncSetAttribute(concat16_fwd_ndhwc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e != cudaSuccess) return (int)e;
        dim3 grid((unsigned)(ntiles * ngroups), (unsigned)H, (unsigned)B);
        concat16_fwd_ndhwc_kernel<<<grid, kCl16Threads, smem, st>>>(l, r, v, (int)C, (int)H, (int)W, (int)Dq, (int)ntiles);
        AZ_LAUNCH_CHECK();
        return 0;
    }
    if (B * 2 * C > 65535 * 32) return AZ_ERR_BAD_ARG;
    const int64_t ngroups = ceil_div(Dq, kF16DG);
    if ((W % 8 == 0) && aligned16(L) && aligned16(R) && aligned16(vol) && 2 * C * ngroups <= 65535) {
        dim3 grid((unsigned)ceil_div(H * (W / 8), 256), (unsigned)(2 * C * ngroups), (unsigned)B);
        concat16_fwd_vec8_kernel<<<grid, 256, 0, st>>>(l, r, v, (int)C, (int)H, (int)W, (int)Dq, (int)ngroups);
        AZ_LAUNCH_CHECK();
        return 0;
    }
    dim3 grid((unsigned)ceil_div(H * W, 256), (unsigned)Dq, (unsigned)(B * 2 * C));
    concat16_fwd_scalar_kernel<<<grid, 256, 0, st>>>(l, r, v, (int)C, (int)H, (int)W, (int)Dq);
    AZ_LAUNCH_CHECK();
    return 0;
}

extern "C" int az_concat_volume_bwd_16(const void* gvol, void* gL, void* gR, int64_t B, int64_t C, int64_t H, int64_t W,
                                       int64_t Dq, int dtype, int channels_last, void* stream) {
    if (!gvol || B <= 0 || C <= 0 || H <= 0 || W <= 0 || Dq <= 0) return AZ_ERR_BAD_ARG;
    if (dtype != AZ_DTYPE_BF16 && dtype != AZ_DTYPE_F16) return AZ_ERR_BAD_ARG;
    if (H * W >= (1ll << 31) / 8 || B > 65535 || 2 * C > 65535) return AZ_ERR_BAD_ARG;
    if (channels_last && ((C % 8) != 0 || !aligned16(gvol) || H > 65535)) return AZ_ERR_BAD_ARG;
    if (channels_last && (size_t)(2 * C) * (kCl16TXB + 2) * sizeof(uint16_t) > 200 * 1024) return AZ_ERR_BAD_ARG;
    if (!gL && !gR) return 0;
    const uint16_t* g = static_cast<const uint16_t*>(gvol);
    uint16_t* l = static_cast<uint16_t*>(gL);
    uint16_t* r = static_cast<uint16_t*>(gR);
    cudaStream_t st = (cudaStream_t)stream;
    return dtype == AZ_DTYPE_BF16 ? concat16_bwd_launch<AZ_DTYPE_BF16>(g, l, r, B, C, H, W, Dq, channels_last != 0, st)
                                  : concat16_bwd_launch<AZ_DTYPE_F16>(g, l, r, B, C, H, W, Dq, channels_last != 0, st);
}
