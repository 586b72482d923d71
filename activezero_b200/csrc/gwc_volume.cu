// Group-wise correlation volume, forward and backward (SURVEY.md §8a row a3).
// NOT IN THE REFERENCE (SURVEY.md fact 1): the definition is GwcNet's,
//   vol[b,g,i,y,x] = (1/cpg) * sum_{c in group g} L[b,c,y,x] * R[b,c,y,x-i]   (x >= i, else 0)
// with cpg = C/G.  Parity is against this repository's own torch restatement (parity unpinned).
//
// Same data movement as the concat volume.  Forward: the cpg right rows of one (b, g, row-run) are
// staged once in shared memory behind a zero prefix; a thread owns one float4 of output columns,
// keeps its cpg left float4 in registers and sweeps the Dq planes with streaming 128-bit stores,
// reading the shifted right window as two aligned float4 + a static register window (one LDS.128
// per channel per four disparities).  Backward: direct 128-bit loads of the gradient planes (three
// aligned float4 per plane: column x for gL, columns x+4m and x+4m+4 for the x+i diagonal of gR),
// left/right rows in shared memory, fixed-order accumulation in registers: gather-style, atomic-free.
//
// The kernels the entry points run at their defaults are templated on the tensor dtype T (float, bf16, fp16; DESIGN.md
// §4.15).  A 16-bit value is widened to fp32 exactly where it is read -- at the register load, or at the LDS from a
// stage that a bulk copy filled with raw 16-bit bytes -- and from there on every instruction is the fp32 kernel's: the
// fmaf chains in the same order, `inv` applied at the same place, fp32 accumulators, the same systolic hand-over.  Each
// 16-bit result is rounded once, to nearest even, at its store, so a 16-bit kernel returns the fp32 kernel's result on
// the widened inputs followed by .to(dtype).
#include <type_traits>

#include "common.cuh"

namespace az {

constexpr int kGwcThreads = 256;

// ---- element access of the templated kernels ----------------------------------------------------------------------
// A quad is four consecutive elements: one 16-byte access in fp32, one 8-byte access in 16 bits (raw type GwcQuad<T>).
// For T = float every helper is the plain access the fp32 kernels always made.
template <typename T> struct GwcQuadT { using type = uint2; };
template <> struct GwcQuadT<float> { using type = float4; };
template <typename T> using GwcQuad = typename GwcQuadT<T>::type;

template <typename T>
__device__ __forceinline__ float4 widen4(const GwcQuad<T>& q) {
    if constexpr (std::is_same<T, float>::value) {
        return q;
    } else if constexpr (std::is_same<T, __nv_bfloat16>::value) {
        return make_float4(__uint_as_float(q.x << 16), __uint_as_float(q.x & 0xffff0000u), __uint_as_float(q.y << 16),
                           __uint_as_float(q.y & 0xffff0000u));
    } else {
        const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&q.x));
        const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&q.y));
        return make_float4(a.x, a.y, b.x, b.y);
    }
}
// one RNE rounding per element; an fp16 value outside the format becomes +-inf, as .to(torch.float16) makes it
template <typename T>
__device__ __forceinline__ GwcQuad<T> narrow4(const float4& v) {
    if constexpr (std::is_same<T, float>::value) {
        return v;
    } else if constexpr (std::is_same<T, __nv_bfloat16>::value) {
        const __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
        return make_uint2(*reinterpret_cast<const uint32_t*>(&a), *reinterpret_cast<const uint32_t*>(&b));
    } else {
        const __half2 a = __floats2half2_rn(v.x, v.y), b = __floats2half2_rn(v.z, v.w);
        return make_uint2(*reinterpret_cast<const uint32_t*>(&a), *reinterpret_cast<const uint32_t*>(&b));
    }
}
// quad k of the row at p (read-only path)
template <typename T>
__device__ __forceinline__ float4 ldg4(const T* p, int k = 0) {
    return widen4<T>(__ldg(reinterpret_cast<const GwcQuad<T>*>(p) + k));
}
template <typename T>
__device__ __forceinline__ void st4(T* p, const float4& v) {
    *reinterpret_cast<GwcQuad<T>*>(p) = narrow4<T>(v);
}
template <typename T>
__device__ __forceinline__ void st4_stream(T* p, const float4& v) {
    __stcs(reinterpret_cast<GwcQuad<T>*>(p), narrow4<T>(v));
}
__device__ __forceinline__ float ldcs_f32(const float* p) { return __ldcs(p); }
__device__ __forceinline__ float ldcs_f32(const __nv_bfloat16* p) { return __bfloat162float(__ldcs(p)); }
__device__ __forceinline__ float ldcs_f32(const __half* p) { return __half2float(__ldcs(p)); }
__device__ __forceinline__ void stcs_from_f32(float* p, float v) { __stcs(p, v); }
__device__ __forceinline__ void stcs_from_f32(__nv_bfloat16* p, float v) { __stcs(p, __float2bfloat16_rn(v)); }
__device__ __forceinline__ void stcs_from_f32(__half* p, float v) { __stcs(p, __float2half_rn(v)); }

// window [k, k+4) of the 8 floats (a, b), k in 1..4 static after unrolling
__device__ __forceinline__ float4 win8(const float4& a, const float4& b, int k) {
    switch (k) {
        case 1: return make_float4(a.y, a.z, a.w, b.x);
        case 2: return make_float4(a.z, a.w, b.x, b.y);
        case 3: return make_float4(a.w, b.x, b.y, b.z);
        default: return b;
    }
}

// grid = (ceil(H*W/4 / 256), G, B); one float4 position per thread.
// smem: Rs[CPG][rows_cap][pad + W], ONE copy per channel behind a zero prefix of pad >= Dq+4
// floats.  The shift by i = 4m+r is the window [4-r, 8-r) of two aligned float4 (A at x-4m-4, B at
// x-4m); B of step m+1 is A of step m, so each thread issues one LDS.128 per channel per FOUR
// disparities and selects the window with static register indices.
template <int CPG>
__global__ void __launch_bounds__(kGwcThreads) gwc_fwd_vec4_kernel(const float* __restrict__ L,
                                                                  const float* __restrict__ R,
                                                                  float* __restrict__ vol, int C, int H, int W,
                                                                  int Dq, int pad, int rows_cap) {
    extern __shared__ __align__(16) float smem[];
    const int W4 = W >> 2;
    const int g = blockIdx.y, b = blockIdx.z, G = gridDim.y;
    const int p0 = blockIdx.x * kGwcThreads;
    const int pend = min(p0 + kGwcThreads, H * W4);
    const size_t HW = (size_t)H * W;
    const int y_first = p0 / W4, y_last = (pend - 1) / W4, nrows = y_last - y_first + 1;
    const int S = pad + W, S4 = S >> 2, pad4 = pad >> 2;
    const int ch_stride = rows_cap * S;
    const float* Lg = L + ((size_t)b * C + (size_t)g * CPG) * HW;
    const float* Rg = R + ((size_t)b * C + (size_t)g * CPG) * HW;

    for (int t = threadIdx.x; t < CPG * nrows * S4; t += kGwcThreads) {
        const int c = t / (nrows * S4), rem = t - c * nrows * S4;
        const int y = rem / S4, q = rem - y * S4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (q >= pad4)
            v = __ldg(reinterpret_cast<const float4*>(Rg + (size_t)c * HW + (size_t)(y_first + y) * W) + (q - pad4));
        reinterpret_cast<float4*>(smem + c * ch_stride + y * S)[q] = v;
    }
    __syncthreads();

    const int pp = p0 + threadIdx.x;
    if (pp >= pend) return;
    const int y = pp / W4, x = (pp - y * W4) * 4;
    float4 l[CPG], Bw[CPG];
    const float* sp = smem + (y - y_first) * S + pad + x;
#pragma unroll
    for (int c = 0; c < CPG; ++c) {
        l[c] = __ldg(reinterpret_cast<const float4*>(Lg + (size_t)c * HW + (size_t)pp * 4));
        Bw[c] = *reinterpret_cast<const float4*>(sp + c * ch_stride);
    }
    float* out = vol + ((size_t)b * G + g) * Dq * HW + (size_t)pp * 4;
    const float inv = 1.0f / (float)CPG;
    for (int m4 = 0; m4 < Dq; m4 += 4) {
        float4 A[CPG];
#pragma unroll
        for (int c = 0; c < CPG; ++c) A[c] = *reinterpret_cast<const float4*>(sp + c * ch_stride - m4 - 4);
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            if (m4 + r < Dq) {
                float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                for (int c = 0; c < CPG; ++c) {
                    const float4 w = win8(A[c], Bw[c], 4 - r);
                    acc.x = fmaf(l[c].x, w.x, acc.x);
                    acc.y = fmaf(l[c].y, w.y, acc.y);
                    acc.z = fmaf(l[c].z, w.z, acc.z);
                    acc.w = fmaf(l[c].w, w.w, acc.w);
                }
                acc.x *= inv; acc.y *= inv; acc.z *= inv; acc.w *= inv;
                st_stream(reinterpret_cast<float4*>(out + (size_t)(m4 + r) * HW), acc);
            }
        }
#pragma unroll
        for (int c = 0; c < CPG; ++c) Bw[c] = A[c];
    }
}


// ------------------------------------------------------------------------------------------
// forward, short-lived CTAs (round 2; the kernel above swept all Dq planes per CTA and reached
// 0.50-0.73 of the measured peak).  Same shape as the concat forward that sits at the store-stream
// ceiling: a CTA owns 256 float4 positions of one (b, group) and writes `DG` consecutive disparity
// planes; the left quads stay in registers, the shifted right window of plane i = 4m + r is the static
// register window [4-r, 8-r) of two aligned quads read straight from the L2-resident feature plane
// (B of step m+1 is A of step m).  No shared memory, no barrier.
// grid = (ceil(H*W/4 / 256), G * ceil(Dq/DG), B)
// ------------------------------------------------------------------------------------------
template <typename T, int CPG>
__global__ void __launch_bounds__(kGwcThreads) gwc_fwd_planes_kernel(const T* __restrict__ L, const T* __restrict__ R,
                                                                    T* __restrict__ vol, int C, int G, int H, int W,
                                                                    int Dq, int DG, int ngroups) {
    const int W4 = W >> 2;
    const int g = blockIdx.y / ngroups, dg = blockIdx.y - g * ngroups, b = blockIdx.z;
    const int i0 = dg * DG, i1 = min(Dq, i0 + DG);
    const int pp = blockIdx.x * kGwcThreads + threadIdx.x;
    if (pp >= H * W4) return;
    const int x = (pp % W4) * 4;
    const size_t HW = (size_t)H * W;
    const T* Lg = L + ((size_t)b * C + (size_t)g * CPG) * HW + (size_t)pp * 4;
    const T* Rg = R + ((size_t)b * C + (size_t)g * CPG) * HW + (size_t)pp * 4;
    const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
    const float inv = 1.0f / (float)CPG;
    float4 l[CPG], Bw[CPG];
#pragma unroll
    for (int c = 0; c < CPG; ++c) {
        float4 t = ldg4(Lg + (size_t)c * HW);
        l[c] = make_float4(t.x * inv, t.y * inv, t.z * inv, t.w * inv);
        Bw[c] = (x - i0 >= 0) ? ldg4(Rg + (size_t)c * HW - i0) : zero;
    }
    T* out = vol + ((size_t)b * G + g) * Dq * HW + (size_t)pp * 4;
    for (int m4 = i0; m4 < i1; m4 += 4) {
        float4 A[CPG];
#pragma unroll
        for (int c = 0; c < CPG; ++c) {
            if constexpr (std::is_same<T, float>::value) {
                A[c] = (x - m4 - 4 >= 0) ? ldg4(Rg + (size_t)c * HW - m4 - 4) : zero;
            } else {  // select the raw quad, then widen (a select after the widening made ptxas spill)
                const uint2 a = (x - m4 - 4 >= 0) ? __ldg(reinterpret_cast<const uint2*>(Rg + (size_t)c * HW - m4 - 4))
                                                  : make_uint2(0u, 0u);
                A[c] = widen4<T>(a);
            }
        }
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            if (m4 + r < i1) {
                float4 acc = zero;
#pragma unroll
                for (int c = 0; c < CPG; ++c) {
                    const float4 w = win8(A[c], Bw[c], 4 - r);
                    acc.x = fmaf(l[c].x, w.x, acc.x);
                    acc.y = fmaf(l[c].y, w.y, acc.y);
                    acc.z = fmaf(l[c].z, w.z, acc.z);
                    acc.w = fmaf(l[c].w, w.w, acc.w);
                }
                st4_stream(out + (size_t)(m4 + r) * HW, acc);
            }
        }
#pragma unroll
        for (int c = 0; c < CPG; ++c) Bw[c] = A[c];
    }
}

// scalar fallback, any shape.  grid = (ceil(H*W/256), Dq, B*G)
template <typename T>
__global__ void __launch_bounds__(256) gwc_fwd_scalar_kernel(const T* __restrict__ L, const T* __restrict__ R,
                                                             T* __restrict__ vol, int C, int G, int H, int W, int Dq) {
    const int hw = blockIdx.x * 256 + threadIdx.x;
    if (hw >= H * W) return;
    const int i = blockIdx.y, bg = blockIdx.z, b = bg / G, g = bg - b * G;
    const int cpg = C / G, x = hw % W;
    const size_t HW = (size_t)H * W;
    float acc = 0.f;
    if (x >= i) {
        const T* l = L + ((size_t)b * C + (size_t)g * cpg) * HW + hw;
        const T* r = R + ((size_t)b * C + (size_t)g * cpg) * HW + hw - i;
        for (int c = 0; c < cpg; ++c) acc = fmaf(ld_f32(l + (size_t)c * HW), ld_f32(r + (size_t)c * HW), acc);
        acc *= 1.0f / (float)cpg;
    }
    stcs_from_f32(vol + (((size_t)bg * Dq + i) * H) * W + hw, acc);
}

// window [k, k+4) of the 8 floats (a, b), k in 0..4
__device__ __forceinline__ float4 win8k(const float4& a, const float4& b, int k) { return k == 0 ? a : win8(a, b, k); }

__device__ __forceinline__ void fma4(float4& acc, const float4& u, const float4& v) {
    acc.x = fmaf(u.x, v.x, acc.x);
    acc.y = fmaf(u.y, v.y, acc.y);
    acc.z = fmaf(u.z, v.z, acc.z);
    acc.w = fmaf(u.w, v.w, acc.w);
}

// ------------------------------------------------------------------------------------------
// backward, direct path (W % 4 == 0): grid = (ceil(H*W/4 / 256), G * (CPG/CPT), B).
// A thread owns one float4 of columns for CPT channels of its group.
//   gL[c,x] = inv * sum_{i<=x} g[i,x] * R[c,x-i];   gR[c,x] = inv * sum_{x+i<W} g[i,x+i] * L[c,x+i]
// smem: Ls[CPT][rows_cap][W + tail] (zero tail) | Rs[CPT][rows_cap][pad + W] (zero prefix)
// ------------------------------------------------------------------------------------------
template <typename T, int CPG, int CPT>
__global__ void __launch_bounds__(kGwcThreads, 3) gwc_bwd_direct_kernel(const T* __restrict__ gvol,
                                                                       const T* __restrict__ L,
                                                                       const T* __restrict__ R,
                                                                       T* __restrict__ gL, T* __restrict__ gR,
                                                                       int C, int G, int H, int W, int Dq, int pad,
                                                                       int rows_cap) {
    extern __shared__ __align__(16) float smem[];
    constexpr int NCH = CPG / CPT;
    const int W4 = W >> 2;
    const int g = blockIdx.y / NCH, chunk = blockIdx.y - g * NCH, b = blockIdx.z;
    const int p0 = blockIdx.x * kGwcThreads;
    const int pend = min(p0 + kGwcThreads, H * W4);
    const size_t HW = (size_t)H * W;
    const int y_first = p0 / W4, y_last = (pend - 1) / W4, nrows = y_last - y_first + 1;
    const int S = pad + W, S4 = S >> 2, pad4 = pad >> 2;  // same stride for both arrays
    const int ch_stride = rows_cap * S;
    float* Ls = smem;
    float* Rs = smem + CPT * ch_stride;
    const size_t cbase = ((size_t)b * C + (size_t)g * CPG + (size_t)chunk * CPT) * HW;

    for (int t = threadIdx.x; t < CPT * nrows * S4; t += kGwcThreads) {
        const int c = t / (nrows * S4), rem = t - c * nrows * S4;
        const int y = rem / S4, q = rem - y * S4;
        const size_t row = cbase + (size_t)c * HW + (size_t)(y_first + y) * W;
        float4 rv = make_float4(0.f, 0.f, 0.f, 0.f), lv = rv;
        if (q >= pad4) rv = ldg4(R + row, q - pad4);
        if (q < W4) lv = ldg4(L + row, q);
        reinterpret_cast<float4*>(Rs + c * ch_stride + y * S)[q] = rv;
        reinterpret_cast<float4*>(Ls + c * ch_stride + y * S)[q] = lv;
    }
    __syncthreads();

    const int pp = p0 + threadIdx.x;
    if (pp >= pend) return;
    const int y = pp / W4, x = (pp - y * W4) * 4;
    const float* rp = Rs + (y - y_first) * S + pad + x;
    const float* lp = Ls + (y - y_first) * S + x;
    const T* gp = gvol + ((size_t)b * G + g) * Dq * HW + (size_t)pp * 4;
    const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 aL[CPT], aR[CPT], RB[CPT], LA[CPT];
#pragma unroll
    for (int c = 0; c < CPT; ++c) {
        aL[c] = zero;
        aR[c] = zero;
        RB[c] = *reinterpret_cast<const float4*>(rp + c * ch_stride);
        LA[c] = *reinterpret_cast<const float4*>(lp + c * ch_stride);
    }
    for (int m4 = 0; m4 < Dq; m4 += 4) {
        float4 gl[4], ga[4], gb[4];
        const bool inA = (x + m4) < W, inB = (x + m4 + 4) < W;
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int i = m4 + r;
            const T* q = gp + (size_t)i * HW;
            const bool on = i < Dq;
            gl[r] = (on && i <= x + 3) ? ldg4(q) : zero;
            ga[r] = (on && inA) ? ldg4(q + m4) : zero;
            gb[r] = (on && inB) ? ldg4(q + m4 + 4) : zero;
        }
        float4 RA[CPT], LB[CPT];
#pragma unroll
        for (int c = 0; c < CPT; ++c) {
            RA[c] = *reinterpret_cast<const float4*>(rp + c * ch_stride - m4 - 4);
            LB[c] = *reinterpret_cast<const float4*>(lp + c * ch_stride + m4 + 4);
        }
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const float4 gw = win8k(ga[r], gb[r], r);
#pragma unroll
            for (int c = 0; c < CPT; ++c) {
                fma4(aL[c], gl[r], win8(RA[c], RB[c], 4 - r));
                fma4(aR[c], gw, win8k(LA[c], LB[c], r));
            }
        }
#pragma unroll
        for (int c = 0; c < CPT; ++c) {
            RB[c] = RA[c];
            LA[c] = LB[c];
        }
    }
    const float inv = 1.0f / (float)CPG;
#pragma unroll
    for (int c = 0; c < CPT; ++c) {
        const size_t o = cbase + (size_t)c * HW + (size_t)pp * 4;
        if (gL != nullptr) st4(gL + o, make_float4(aL[c].x * inv, aL[c].y * inv, aL[c].z * inv, aL[c].w * inv));
        if (gR != nullptr) st4(gR + o, make_float4(aR[c].x * inv, aR[c].y * inv, aR[c].z * inv, aR[c].w * inv));
    }
}


// ------------------------------------------------------------------------------------------
// backward, one pass over the gradient volume (round 2; the direct kernel above re-read the
// volume once per channel pair and reached 0.33-0.45 of the measured peak).
// One CTA owns one image row y of one (b, group): the Dq gradient rows g[i][y][:], and the CPG left /
// right feature rows, are brought into shared memory with 1-D bulk async copies (TMA, one per row,
// completing on an mbarrier) -- every byte of gvol crosses HBM exactly once -- and both gradients are
// then formed from shared memory in a fixed order (gather-style, atomic-free):
//   gL[c,x] = inv * sum_i g[i,x]   * R[c,x-i]     (R behind a zero prefix)
//   gR[c,x] = inv * sum_i g[i,x+i] * L[c,x+i]     (g and L in front of a zero tail)
// A thread owns one float4 of columns of one side for ALL CPG channels, so a gradient quad is read from
// shared memory once per side.  grid = (H, G, B), 128 threads.
// smem: Gs[Dq][GP] | Ls[CPG][GP] | Rs[CPG][pad + W];  GP = W + Dq + 8 (rounded), pad = Dq + 4 (rounded)
// ------------------------------------------------------------------------------------------
constexpr int kGwcRowThreads = 128;

template <int CPG>
__global__ void __launch_bounds__(kGwcRowThreads) gwc_bwd_row_kernel(const float* __restrict__ gvol,
                                                                    const float* __restrict__ L,
                                                                    const float* __restrict__ R,
                                                                    float* __restrict__ gL, float* __restrict__ gR,
                                                                    int C, int G, int H, int W, int Dq, int GP, int pad) {
    extern __shared__ __align__(16) float smem[];
    __shared__ __align__(8) uint64_t bar;
    float* Gs = smem;
    float* Ls = Gs + (size_t)Dq * GP;
    float* Rs = Ls + (size_t)CPG * GP;
    const int RP = pad + W;
    const int tid = threadIdx.x;
    const int y = blockIdx.x, g = blockIdx.y, b = blockIdx.z;
    const size_t HW = (size_t)H * W;
    const uint32_t row_bytes = (uint32_t)W * 4u;

    if (tid == 0) {
        mbar_init(&bar, 1);
        mbar_fence_init();
        mbar_expect_tx(&bar, row_bytes * (uint32_t)(Dq + 2 * CPG));
    }
    // zero tails / prefix (disjoint from the bulk destinations)
    const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
    const int tailq = (GP - W) >> 2, padq = pad >> 2;
    for (int t = tid; t < (Dq + CPG) * tailq; t += kGwcRowThreads) {
        const int r = t / tailq, q = t - r * tailq;
        reinterpret_cast<float4*>(Gs + (size_t)r * GP + W)[q] = zero;  // Ls rows follow Gs with the same pitch
    }
    for (int t = tid; t < CPG * padq; t += kGwcRowThreads) {
        const int r = t / padq, q = t - r * padq;
        reinterpret_cast<float4*>(Rs + (size_t)r * RP)[q] = zero;
    }
    __syncthreads();
    const float* grow = gvol + ((size_t)b * G + g) * Dq * HW + (size_t)y * W;
    const size_t fbase = ((size_t)b * C + (size_t)g * CPG) * HW + (size_t)y * W;
    for (int r = tid; r < Dq + 2 * CPG; r += kGwcRowThreads) {
        if (r < Dq) bulk_g2s(Gs + (size_t)r * GP, grow + (size_t)r * HW, row_bytes, &bar);
        else if (r < Dq + CPG) bulk_g2s(Ls + (size_t)(r - Dq) * GP, L + fbase + (size_t)(r - Dq) * HW, row_bytes, &bar);
        else bulk_g2s(Rs + (size_t)(r - Dq - CPG) * RP + pad, R + fbase + (size_t)(r - Dq - CPG) * HW, row_bytes, &bar);
    }
    mbar_wait(&bar, 0);

    const int W4 = W >> 2;
    const float inv = 1.0f / (float)CPG;
    for (int task = tid; task < 2 * W4; task += kGwcRowThreads) {
        const bool right = task >= W4;
        const int x = (right ? task - W4 : task) * 4;
        float* gout = right ? gR : gL;
        if (gout == nullptr) continue;
        float4 acc[CPG], A[CPG], Bq[CPG];
#pragma unroll
        for (int c = 0; c < CPG; ++c) acc[c] = zero;
        if (!right) {
            const float* rp = Rs + pad + x;
#pragma unroll
            for (int c = 0; c < CPG; ++c) Bq[c] = *reinterpret_cast<const float4*>(rp + c * RP);
            for (int m4 = 0; m4 < Dq; m4 += 4) {
#pragma unroll
                for (int c = 0; c < CPG; ++c) A[c] = *reinterpret_cast<const float4*>(rp + c * RP - m4 - 4);
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    if (m4 + r < Dq) {
                        const float4 gq = *reinterpret_cast<const float4*>(Gs + (size_t)(m4 + r) * GP + x);
#pragma unroll
                        for (int c = 0; c < CPG; ++c) fma4(acc[c], gq, win8(A[c], Bq[c], 4 - r));
                    }
                }
#pragma unroll
                for (int c = 0; c < CPG; ++c) Bq[c] = A[c];
            }
        } else {
            const float* lp = Ls + x;
#pragma unroll
            for (int c = 0; c < CPG; ++c) A[c] = *reinterpret_cast<const float4*>(lp + c * GP);
            for (int m4 = 0; m4 < Dq; m4 += 4) {
#pragma unroll
                for (int c = 0; c < CPG; ++c) Bq[c] = *reinterpret_cast<const float4*>(lp + c * GP + m4 + 4);
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    if (m4 + r < Dq) {
                        const float* gp = Gs + (size_t)(m4 + r) * GP + x + m4;
                        const float4 ga = *reinterpret_cast<const float4*>(gp);
                        const float4 gb = *reinterpret_cast<const float4*>(gp + 4);
                        const float4 gw = win8k(ga, gb, r);
#pragma unroll
                        for (int c = 0; c < CPG; ++c) fma4(acc[c], gw, win8k(A[c], Bq[c], r));
                    }
                }
#pragma unroll
                for (int c = 0; c < CPG; ++c) A[c] = Bq[c];
            }
        }
#pragma unroll
        for (int c = 0; c < CPG; ++c)
            *reinterpret_cast<float4*>(gout + fbase + (size_t)c * HW + x) =
                make_float4(acc[c].x * inv, acc[c].y * inv, acc[c].z * inv, acc[c].w * inv);
    }
}

// ------------------------------------------------------------------------------------------
// backward, systolic one-pass kernel (round 2, default).  The direct kernel needs every gradient quad in two
// alignments (column x for gL, the x + i diagonal for gR: three 128-bit loads per plane, LSU-bound at 0.46 of the
// HBM peak).  Here a gradient quad g[i][x..x+3] is read ONCE, aligned, and serves both sides:
//   gL[c][x+j]     += g[i][x+j] * R[c][x+j-i]           (own columns; right window = static register window)
//   gR[c][x+j-i]   += g[i][x+j] * L[c][x+j]             (own L quad in registers; the TARGET moves, not the data)
// The accumulator of the target quad Q_k = columns [4k, 4k+4) travels: at step m (planes 4m..4m+3) it sits in the
// thread t = k + m of the row, takes that thread's contributions with j >= r ("high"), moves one thread to the right
// (shfl_up; lane 31 -> lane 0 of the next warp through shared memory) and takes the same thread's contributions
// with j < r ("low").  After ceil(Dq/4) steps thread t holds the finished Q_{t-M}; quads whose walk leaves the row on
// the right are finished early and written by the row's last thread.  Fixed order, atomic-free, deterministic.
//
// Data movement: a CTA owns `rows` = NT/(W/4) whole image rows of one (b, group); its positions are contiguous in
// every plane, so a gradient plane of the CTA is ONE 1-D bulk async copy (TMA, nact*16 bytes), four planes per stage,
// kGwcSysStages stages on mbarriers; the feature rows arrive the same way.  Measured (B=8, 136x240, Dq=48, G=8):
// the kernel is bound by the bytes the stage rings keep in flight (four 128-thread CTAs x 4 stages x 7.7 KB per SM):
// 3 stages 0.67, 4 stages 0.75, 5 stages (left quads read straight into registers) 0.77, and 0.80 once the refill
// copies are spread over four warps, against 0.46 for the direct kernel; 256-thread CTAs 0.73-0.77.  A persistent variant (stage ring running
// across tiles, features one tile ahead) needs a second right-feature buffer, which costs a stage: 0.69.  An L2
// prefetch ahead of the ring (cp.async.bulk.prefetch.L2) made it slower (0.51): the extra requests queue in front of
// the copies the ring waits for.
// grid = (ceil(H / rows), G, B).
// ------------------------------------------------------------------------------------------

// LSM: left rows staged in shared memory (S = 4) or read straight into registers (S = 5: their 8 KB buy a stage)
// 16 bits: the stages, Ls and Rs hold raw 16-bit quads (8 bytes), widened at the LDS; `hand` carries fp32 accumulators.
template <typename T, int CPG, int NT, int S, bool LSM>
__global__ void __launch_bounds__(NT, 512 / NT) gwc_bwd_systolic_kernel(const T* __restrict__ gvol,
                                                                       const T* __restrict__ L,
                                                                       const T* __restrict__ R,
                                                                       T* __restrict__ gL, T* __restrict__ gR,
                                                                       int C, int G, int H, int W, int Dq, int rows) {
    using Q = GwcQuad<T>;
    extern __shared__ __align__(128) float4 stage_smem[];
    Q* stage = reinterpret_cast<Q*>(stage_smem);  // [S][4][NT] | Ls[CPG][NT] | Rs[CPG][NT]
    __shared__ __align__(8) uint64_t full[S];
    __shared__ __align__(8) uint64_t feat_bar;
    __shared__ float4 hand[2][NT / 32 + 1][CPG];  // slot w + 1: lane 31 of warp w; slot 0 stays zero
    __shared__ Q zslot;                           // stands in for the planes >= Dq of the last step
    const int W4 = W >> 2;
    const int g = blockIdx.y, b = blockIdx.z;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int y0 = blockIdx.x * rows;
    const int nact = min(rows, H - y0) * W4;  // threads that own a quad
    const bool active = tid < nact;
    const int q = tid % W4;
    const bool row_end = q == W4 - 1;
    const size_t HW = (size_t)H * W;
    const size_t p0 = (size_t)y0 * W;  // first float of the CTA's positions within a plane
    const T* gbase = gvol + ((size_t)b * G + g) * Dq * HW + p0;
    const size_t cbase = ((size_t)b * C + (size_t)g * CPG) * HW + p0 + (size_t)tid * 4;
    const int M = (Dq + 3) >> 2;
    const uint32_t plane_bytes = (uint32_t)nact * (uint32_t)sizeof(Q);
    const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);

    auto issue = [&](int m) {  // one thread: the four planes of step m -> stage m % S
        const int s = m % S, np = min(4, Dq - 4 * m);
        mbar_expect_tx(&full[s], plane_bytes * (uint32_t)np);
        for (int r = 0; r < np; ++r)
            bulk_g2s(stage + (size_t)(s * 4 + r) * NT, gbase + (size_t)(4 * m + r) * HW, plane_bytes, &full[s]);
    };
    Q* Ls = stage + (size_t)S * 4 * NT;
    Q* Rs = Ls + (LSM ? (size_t)CPG * NT : 0);
    if (warp == 0) {
        // lane 0 arms the barriers, then the lanes issue the first copies
        if (lane == 0) {
#pragma unroll
            for (int s = 0; s < S; ++s) mbar_init(&full[s], 1);
            mbar_init(&feat_bar, 1);
            mbar_fence_init();
            mbar_expect_tx(&feat_bar, plane_bytes * (uint32_t)((LSM ? 2 : 1) * CPG));
            for (int m = 0; m < min(M, S); ++m)
                mbar_expect_tx(&full[m], plane_bytes * (uint32_t)min(4, Dq - 4 * m));
            if constexpr (std::is_same<T, float>::value) zslot = zero;
            else zslot = make_uint2(0u, 0u);
        }
        __syncwarp();
        const size_t fb = ((size_t)b * C + (size_t)g * CPG) * HW + p0;
        if (lane < 2 * CPG) {
            const int c = lane >> 1;
            if (lane & 1) bulk_g2s(Rs + (size_t)c * NT, R + fb + (size_t)c * HW, plane_bytes, &feat_bar);
            else if (LSM) bulk_g2s(Ls + (size_t)c * NT, L + fb + (size_t)c * HW, plane_bytes, &feat_bar);
        } else if (lane >= 8 && lane - 8 < min(Dq, 4 * S)) {
            const int i = lane - 8;  // plane i -> stage i / 4, slot i % 4
            bulk_g2s(stage + (size_t)i * NT, gbase + (size_t)i * HW, plane_bytes, &full[i >> 2]);
            if constexpr (4 * S > 24) {  // a ring of more than six stages: the 24 lanes take further rounds
                for (int i2 = i + 24; i2 < min(Dq, 4 * S); i2 += 24)
                    bulk_g2s(stage + (size_t)i2 * NT, gbase + (size_t)i2 * HW, plane_bytes, &full[i2 >> 2]);
            }
        }
    }
    if (tid < 2 * CPG) hand[tid / CPG][0][tid % CPG] = zero;
    const float inv = 1.0f / (float)CPG;
    __syncthreads();  // barrier initialisation, zero slots visible
    float4 l[CPG], Bw[CPG], aL[CPG], V[CPG];
    if (!LSM) {
#pragma unroll
        for (int c = 0; c < CPG; ++c)
            l[c] = active ? ldg4(L + cbase + (size_t)c * HW) : zero;
    }
    mbar_wait(&feat_bar, 0);
#pragma unroll
    for (int c = 0; c < CPG; ++c) {
        // threads without a quad read stale shared memory: their values never reach a thread that owns one (the walk
        // only moves right)
        if constexpr (std::is_same<T, float>::value) {
            if (LSM) l[c] = Ls[(size_t)c * NT + tid];
            Bw[c] = Rs[(size_t)c * NT + tid];
        } else {
            if (LSM) l[c] = widen4<T>(Ls[(size_t)c * NT + tid]);
            Bw[c] = widen4<T>(Rs[(size_t)c * NT + tid]);
        }
        aL[c] = zero;
        V[c] = zero;
    }
    const int np_last = Dq - 4 * (M - 1);

#pragma unroll 2
    for (int m = 0; m < M; ++m) {
        const int s = m % S;
        const int np = (m == M - 1) ? np_last : 4;
        mbar_wait(&full[s], (uint32_t)((m / S) & 1));
        float4 gq[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) gq[r] = widen4<T>(*((r < np) ? stage + (size_t)(s * 4 + r) * NT + tid : &zslot));
        float4 A[CPG];
#pragma unroll
        for (int c = 0; c < CPG; ++c) {
            if constexpr (std::is_same<T, float>::value) A[c] = (q - m - 1 >= 0) ? Rs[(size_t)c * NT + tid - m - 1] : zero;
            else A[c] = (q - m - 1 >= 0) ? widen4<T>(Rs[(size_t)c * NT + tid - m - 1]) : zero;
        }
#pragma unroll
        for (int c = 0; c < CPG; ++c) {
            // gL: own columns; gR "high" part: targets j - r >= 0 of the quad this thread holds
            fma4(aL[c], gq[0], Bw[c]);
            fma4(V[c], gq[0], l[c]);
            fma4(aL[c], gq[1], win8(A[c], Bw[c], 3));
            V[c].x = fmaf(gq[1].y, l[c].y, V[c].x);
            V[c].y = fmaf(gq[1].z, l[c].z, V[c].y);
            V[c].z = fmaf(gq[1].w, l[c].w, V[c].z);
            fma4(aL[c], gq[2], win8(A[c], Bw[c], 2));
            V[c].x = fmaf(gq[2].z, l[c].z, V[c].x);
            V[c].y = fmaf(gq[2].w, l[c].w, V[c].y);
            fma4(aL[c], gq[3], win8(A[c], Bw[c], 1));
            V[c].x = fmaf(gq[3].w, l[c].w, V[c].x);
        }
        if (row_end) {
            // the walk of Q_{W4-1-m} ends here: finished.  Hand a zero to the first thread of the next row.
            if (active && q - m >= 0 && gR != nullptr) {
#pragma unroll
                for (int c = 0; c < CPG; ++c)
                    st4(gR + cbase + (size_t)c * HW - (size_t)(4 * m),
                        make_float4(V[c].x * inv, V[c].y * inv, V[c].z * inv, V[c].w * inv));
            }
#pragma unroll
            for (int c = 0; c < CPG; ++c) V[c] = zero;
        }
        if (lane == 31) {
#pragma unroll
            for (int c = 0; c < CPG; ++c) hand[m & 1][warp + 1][c] = V[c];
        }
        __syncthreads();  // hand-over slots written; every thread is done with stage s
        // refill of the stage just released (step m + S): the arm goes with warp 0, the four plane copies are issued by
        // lane 0 of warps 0..3, one each -- four copies from ONE thread delay that warp by their issue cost every step
        // and the other warps then wait for it at the next barrier
        if (lane == 0 && warp < 4 && m + S < M) {
            const int mn = m + S, np2 = min(4, Dq - 4 * mn);
            if (warp == 0) mbar_expect_tx(&full[s], plane_bytes * (uint32_t)np2);
            if (warp < np2)
                bulk_g2s(stage + (size_t)(s * 4 + warp) * NT, gbase + (size_t)(4 * mn + warp) * HW, plane_bytes, &full[s]);
        }
#pragma unroll
        for (int c = 0; c < CPG; ++c) {
            float4 rv;
            rv.x = __shfl_up_sync(0xffffffffu, V[c].x, 1);
            rv.y = __shfl_up_sync(0xffffffffu, V[c].y, 1);
            rv.z = __shfl_up_sync(0xffffffffu, V[c].z, 1);
            rv.w = __shfl_up_sync(0xffffffffu, V[c].w, 1);
            if (lane == 0) rv = hand[m & 1][warp][c];
            // gR "low" part of this step: targets 4 + j - r of the quad that has just arrived
            rv.w = fmaf(gq[1].x, l[c].x, rv.w);
            rv.z = fmaf(gq[2].x, l[c].x, rv.z);
            rv.w = fmaf(gq[2].y, l[c].y, rv.w);
            rv.y = fmaf(gq[3].x, l[c].x, rv.y);
            rv.z = fmaf(gq[3].y, l[c].y, rv.z);
            rv.w = fmaf(gq[3].z, l[c].z, rv.w);
            V[c] = rv;
            Bw[c] = A[c];
        }
    }
    if (!active) return;
#pragma unroll
    for (int c = 0; c < CPG; ++c) {
        if (gL != nullptr) st4(gL + cbase + (size_t)c * HW, make_float4(aL[c].x * inv, aL[c].y * inv, aL[c].z * inv, aL[c].w * inv));
        if (gR != nullptr && q - M >= 0)
            st4(gR + cbase + (size_t)c * HW - (size_t)(4 * M), make_float4(V[c].x * inv, V[c].y * inv, V[c].z * inv, V[c].w * inv));
    }
}

// scalar fallback: one thread per (b, c, y, x).  grid = (ceil(H*W/256), C, B)
template <typename T>
__global__ void __launch_bounds__(256) gwc_bwd_scalar_kernel(const T* __restrict__ gvol, const T* __restrict__ L,
                                                             const T* __restrict__ R, T* __restrict__ gL,
                                                             T* __restrict__ gR, int C, int G, int H, int W, int Dq) {
    const int hw = blockIdx.x * 256 + threadIdx.x;
    if (hw >= H * W) return;
    const int c = blockIdx.y, b = blockIdx.z;
    const int cpg = C / G, g = c / cpg, x = hw % W;
    const size_t HW = (size_t)H * W;
    const T* gv = gvol + ((size_t)b * G + g) * Dq * HW + hw;
    const T* l = L + ((size_t)b * C + c) * HW + hw;
    const T* r = R + ((size_t)b * C + c) * HW + hw;
    float aL = 0.f, aR = 0.f;
    for (int i = 0; i < Dq; ++i) {
        if (i <= x) aL = fmaf(ldcs_f32(gv + (size_t)i * HW), ld_f32(r - i), aL);
        if (x + i < W) aR = fmaf(ldcs_f32(gv + (size_t)i * HW + i), ld_f32(l + i), aR);
    }
    const float inv = 1.0f / (float)cpg;
    if (gL != nullptr) st_from_f32(gL + ((size_t)b * C + c) * HW + hw, aL * inv);
    if (gR != nullptr) st_from_f32(gR + ((size_t)b * C + c) * HW + hw, aR * inv);
}

// The 16-bit forms of the kernels follow the fp32 selection at its defaults and read no AZ_GWC_* knob.  Where a 16-bit
// alignment rule excludes the kernel the fp32 entry point would run, a kernel with the same summation order runs:
//   forward : the planes kernel pre-scales the left quads by inv = 1/cpg, a power of two for the cpg it serves, which
//             commutes with every rounding outside fp32's subnormal range; the scalar kernel (sum of cpg products from
//             zero in ascending c, then *inv -- the order of the fp32 grid-overflow kernel gwc_fwd_vec4_kernel) therefore
//             returns the same values;
//   backward: the systolic, direct and scalar kernels all sum the terms g * feature in ascending i from zero and scale by
//             inv once at the end, so any of them returns the same gradient.
// Stage ring of the 16-bit systolic backward.  A 16-bit stage holds half the bytes of an fp32 one, yet at config 2 the
// 16-bit kernel takes the fp32 kernel's time with 5 or 6 stages and is slower with 8 or 10 (benchmarks/micro/
// gwc16_stages.cu, DESIGN.md §4.15): it is bound by the per-step instructions it shares with the fp32 kernel, not by the
// bytes in flight, so it keeps the fp32 ring.
constexpr int kGwcSys16Stages = 5;

inline bool aligned_to(const void* p, size_t n) { return (reinterpret_cast<uintptr_t>(p) % n) == 0; }

template <typename T, int CPG>
static int launch_gwc_fwd(const T* L, const T* R, T* vol, int B, int C, int G, int H, int W, int Dq, cudaStream_t st,
                          bool* done) {
    constexpr bool f32 = std::is_same<T, float>::value;
    const int W4 = W / 4;
    *done = false;
    // planes per CTA; 0 = round-1 kernel (all planes per CTA, rows in shared memory)
    int DG = f32 ? tuning("AZ_GWC_DG", 16) : 16;
    if (DG > 0) {
        DG = (DG + 3) & ~3;
        const int64_t ngroups = ceil_div(Dq, DG);
        if ((int64_t)G * ngroups <= 65535) {
            dim3 grid((unsigned)ceil_div((int64_t)H * W4, kGwcThreads), (unsigned)(G * ngroups), (unsigned)B);
            gwc_fwd_planes_kernel<T, CPG><<<grid, kGwcThreads, 0, st>>>(L, R, vol, C, G, H, W, Dq, DG, (int)ngroups);
            *done = true;
            return (int)cudaGetLastError();
        }
    }
    if constexpr (!f32) {
        return 0;  // grid overflow: the scalar kernel
    } else {
        const int pad = (Dq + 3) / 4 * 4 + 4;
        const int rows_cap = (kGwcThreads + W4 - 1) / W4 + 1;
        const size_t smem = (size_t)CPG * rows_cap * (pad + W) * sizeof(float);
        if (smem > 200 * 1024) return 0;
        cudaError_t e = cudaFuncSetAttribute(gwc_fwd_vec4_kernel<CPG>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             200 * 1024);
        if (e != cudaSuccess) return (int)e;
        dim3 grid((unsigned)ceil_div((int64_t)H * W4, kGwcThreads), (unsigned)G, (unsigned)B);
        gwc_fwd_vec4_kernel<CPG><<<grid, kGwcThreads, smem, st>>>(L, R, vol, C, H, W, Dq, pad, rows_cap);
        *done = true;
        return (int)cudaGetLastError();
    }
}

// systolic_ok: the bases and the row length suit the systolic kernel's bulk copies (16-byte addresses and sizes)
template <typename T, int CPG>
static int launch_gwc_bwd(const T* gvol, const T* L, const T* R, T* gL, T* gR, int B, int C, int G, int H, int W, int Dq,
                          bool systolic_ok, cudaStream_t st, bool* done) {
    constexpr bool f32 = std::is_same<T, float>::value;
    constexpr int CPT = CPG >= 2 ? 2 : 1;
    *done = false;
    const int variant = f32 ? tuning("AZ_GWC_BWD", 2) : 2;  // 2 = systolic one-pass (default), 1 = TMA row kernel, 0 = direct
    if (variant == 2 && systolic_ok && CPG <= 4 && W / 4 <= kGwcThreads && G <= 65535) {
        constexpr int K = CPG <= 4 ? CPG : 1;
        const int W4 = W / 4;
        // 128-thread CTAs (four per SM) hide each other's pipeline fill better than two of 256
        const bool small = W4 <= 128 && (!f32 || tuning("AZ_GWC_BWD_NT", 128) == 128);
        const int nt = small ? 128 : 256, rows = nt / W4;
        const int64_t gx = ceil_div(H, rows);
        if (gx <= 0x7fffffff) {
            void (*kern)(const T*, const T*, const T*, T*, T*, int, int, int, int, int, int);
            size_t smem_sys;
            if constexpr (f32) {
                const bool five = tuning("AZ_GWC_BWD_STAGES", 5) == 5;
                smem_sys = (size_t)(five ? 5 * 4 + K : 4 * 4 + 2 * K) * nt * sizeof(float4);
                kern = small ? (five ? gwc_bwd_systolic_kernel<T, K, 128, 5, false> : gwc_bwd_systolic_kernel<T, K, 128, 4, true>)
                             : (five ? gwc_bwd_systolic_kernel<T, K, 256, 5, false> : gwc_bwd_systolic_kernel<T, K, 256, 4, true>);
            } else {
                smem_sys = (size_t)(kGwcSys16Stages * 4 + K) * nt * sizeof(GwcQuad<T>);
                kern = small ? gwc_bwd_systolic_kernel<T, K, 128, kGwcSys16Stages, false>
                             : gwc_bwd_systolic_kernel<T, K, 256, kGwcSys16Stages, false>;
            }
            cudaError_t es = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_sys);
            if (es != cudaSuccess) return (int)es;
            dim3 grid((unsigned)gx, (unsigned)G, (unsigned)B);
            kern<<<grid, nt, smem_sys, st>>>(gvol, L, R, gL, gR, C, G, H, W, Dq, rows);
            *done = true;
            return (int)cudaGetLastError();
        }
    }
    if constexpr (f32) {
        if (variant == 1 && H <= 65535) {  // one-pass row kernel (TMA bulk staging)
            const int padr = (Dq + 3) / 4 * 4 + 4, GP = (W + Dq + 8 + 3) & ~3;
            const size_t smem_row = ((size_t)(Dq + CPG) * GP + (size_t)CPG * (padr + W)) * sizeof(float);
            if (smem_row <= 200 * 1024 && (size_t)(Dq + 2 * CPG) * W * 4 < (1u << 20)) {
                cudaError_t er = cudaFuncSetAttribute(gwc_bwd_row_kernel<CPG>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                      200 * 1024);
                if (er != cudaSuccess) return (int)er;
                dim3 grid((unsigned)H, (unsigned)G, (unsigned)B);
                gwc_bwd_row_kernel<CPG><<<grid, kGwcRowThreads, smem_row, st>>>(gvol, L, R, gL, gR, C, G, H, W, Dq, GP, padr);
                *done = true;
                return (int)cudaGetLastError();
            }
        }
    }
    const int W4 = W / 4, pad = (Dq + 3) / 4 * 4 + 4;
    const int rows_cap = (kGwcThreads + W4 - 1) / W4 + 1;
    const size_t smem = (size_t)2 * CPT * rows_cap * (pad + W) * sizeof(float);  // rows staged widened to fp32
    if (smem > 100 * 1024 || (long long)G * (CPG / CPT) > 65535) return 0;
    cudaError_t e = cudaFuncSetAttribute(gwc_bwd_direct_kernel<T, CPG, CPT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         100 * 1024);
    if (e != cudaSuccess) return (int)e;
    dim3 grid((unsigned)ceil_div((int64_t)H * W4, kGwcThreads), (unsigned)(G * (CPG / CPT)), (unsigned)B);
    gwc_bwd_direct_kernel<T, CPG, CPT><<<grid, kGwcThreads, smem, st>>>(gvol, L, R, gL, gR, C, G, H, W, Dq, pad, rows_cap);
    *done = true;
    return (int)cudaGetLastError();
}

// Kernel selection shared by the fp32 and 16-bit entry points (arguments already checked).  The quad kernels need
// W % 4 == 0 and quad-aligned bases (16 bytes in fp32, 8 bytes in 16 bits); everything else runs the scalar kernels.
template <typename T>
static int gwc_fwd(const T* L, const T* R, T* vol, int64_t B, int64_t C, int64_t H, int64_t W, int64_t Dq, int64_t G,
                   cudaStream_t st) {
    const size_t qb = sizeof(GwcQuad<T>);
    const int64_t cpg = C / G;
    if ((W % 4 == 0) && aligned_to(L, qb) && aligned_to(R, qb) && aligned_to(vol, qb)) {
        bool done = false;
        int rc = 0;
        switch (cpg) {
            case 1: rc = launch_gwc_fwd<T, 1>(L, R, vol, (int)B, (int)C, (int)G, (int)H, (int)W, (int)Dq, st, &done); break;
            case 2: rc = launch_gwc_fwd<T, 2>(L, R, vol, (int)B, (int)C, (int)G, (int)H, (int)W, (int)Dq, st, &done); break;
            case 4: rc = launch_gwc_fwd<T, 4>(L, R, vol, (int)B, (int)C, (int)G, (int)H, (int)W, (int)Dq, st, &done); break;
            case 8: rc = launch_gwc_fwd<T, 8>(L, R, vol, (int)B, (int)C, (int)G, (int)H, (int)W, (int)Dq, st, &done); break;
            default: break;
        }
        if (rc != 0) return rc;
        if (done) return 0;
    }
    if (Dq > 65535 || B * G > 65535) return AZ_ERR_BAD_ARG;
    dim3 grid((unsigned)ceil_div(H * W, 256), (unsigned)Dq, (unsigned)(B * G));
    gwc_fwd_scalar_kernel<T><<<grid, 256, 0, st>>>(L, R, vol, (int)C, (int)G, (int)H, (int)W, (int)Dq);
    AZ_LAUNCH_CHECK();
    return 0;
}

template <typename T>
static int gwc_bwd(const T* gvol, const T* L, const T* R, T* gL, T* gR, int64_t B, int64_t C, int64_t H, int64_t W,
                   int64_t Dq, int64_t G, cudaStream_t st) {
    const size_t qb = sizeof(GwcQuad<T>);
    const int64_t cpg = C / G;
    auto all_aligned = [&](size_t n) {
        return aligned_to(gvol, n) && aligned_to(L, n) && aligned_to(R, n) && (!gL || aligned_to(gL, n)) &&
               (!gR || aligned_to(gR, n));
    };
    if ((W % 4 == 0) && all_aligned(qb)) {
        // 16 bits: a CTA's plane run of nact = rows * W/4 quads is a multiple of 16 bytes when W % 8 == 0
        const bool systolic_ok = std::is_same<T, float>::value || ((W % 8 == 0) && all_aligned(16));
        bool done = false;
        int rc = 0;
        switch (cpg) {
            case 1: rc = launch_gwc_bwd<T, 1>(gvol, L, R, gL, gR, (int)B, (int)C, (int)G, (int)H, (int)W, (int)Dq, systolic_ok, st, &done); break;
            case 2: rc = launch_gwc_bwd<T, 2>(gvol, L, R, gL, gR, (int)B, (int)C, (int)G, (int)H, (int)W, (int)Dq, systolic_ok, st, &done); break;
            case 4: rc = launch_gwc_bwd<T, 4>(gvol, L, R, gL, gR, (int)B, (int)C, (int)G, (int)H, (int)W, (int)Dq, systolic_ok, st, &done); break;
            case 8: rc = launch_gwc_bwd<T, 8>(gvol, L, R, gL, gR, (int)B, (int)C, (int)G, (int)H, (int)W, (int)Dq, systolic_ok, st, &done); break;
            default: break;
        }
        if (rc != 0) return rc;
        if (done) return 0;
    }
    dim3 grid((unsigned)ceil_div(H * W, 256), (unsigned)C, (unsigned)B);
    gwc_bwd_scalar_kernel<T><<<grid, 256, 0, st>>>(gvol, L, R, gL, gR, (int)C, (int)G, (int)H, (int)W, (int)Dq);
    AZ_LAUNCH_CHECK();
    return 0;
}

}  // namespace az

using namespace az;

extern "C" int az_gwc_volume_fwd(const float* L, const float* R, float* vol, int64_t B, int64_t C, int64_t H,
                                 int64_t W, int64_t Dq, int64_t G, void* stream) {
    if (!L || !R || !vol || B <= 0 || C <= 0 || H <= 0 || W <= 0 || Dq <= 0 || G <= 0 || C % G != 0)
        return AZ_ERR_BAD_ARG;
    if (H * W >= (1ll << 31) / 4 || B > 65535 || G > 65535) return AZ_ERR_BAD_ARG;
    return gwc_fwd(L, R, vol, B, C, H, W, Dq, G, (cudaStream_t)stream);
}

extern "C" int az_gwc_volume_bwd(const float* gvol, const float* L, const float* R, float* gL, float* gR, int64_t B,
                                 int64_t C, int64_t H, int64_t W, int64_t Dq, int64_t G, void* stream) {
    if (!gvol || !L || !R || B <= 0 || C <= 0 || H <= 0 || W <= 0 || Dq <= 0 || G <= 0 || C % G != 0)
        return AZ_ERR_BAD_ARG;
    if (H * W >= (1ll << 31) / 4 || B > 65535 || C > 65535 || H > 65535) return AZ_ERR_BAD_ARG;
    if (!gL && !gR) return 0;
    return gwc_bwd(gvol, L, R, gL, gR, B, C, H, W, Dq, G, (cudaStream_t)stream);
}

extern "C" int az_gwc_volume_fwd_16(const void* L, const void* R, void* vol, int64_t B, int64_t C, int64_t H, int64_t W,
                                    int64_t Dq, int64_t G, int dtype, void* stream) {
    if (dtype != AZ_DTYPE_BF16 && dtype != AZ_DTYPE_F16) return AZ_ERR_BAD_ARG;
    if (!L || !R || !vol || B <= 0 || C <= 0 || H <= 0 || W <= 0 || Dq <= 0 || G <= 0 || C % G != 0)
        return AZ_ERR_BAD_ARG;
    if (H * W >= (1ll << 31) / 4 || B > 65535 || G > 65535) return AZ_ERR_BAD_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == AZ_DTYPE_BF16)
        return gwc_fwd(static_cast<const __nv_bfloat16*>(L), static_cast<const __nv_bfloat16*>(R),
                       static_cast<__nv_bfloat16*>(vol), B, C, H, W, Dq, G, st);
    return gwc_fwd(static_cast<const __half*>(L), static_cast<const __half*>(R), static_cast<__half*>(vol), B, C, H, W,
                   Dq, G, st);
}

extern "C" int az_gwc_volume_bwd_16(const void* gvol, const void* L, const void* R, void* gL, void* gR, int64_t B,
                                    int64_t C, int64_t H, int64_t W, int64_t Dq, int64_t G, int dtype, void* stream) {
    if (dtype != AZ_DTYPE_BF16 && dtype != AZ_DTYPE_F16) return AZ_ERR_BAD_ARG;
    if (!gvol || !L || !R || B <= 0 || C <= 0 || H <= 0 || W <= 0 || Dq <= 0 || G <= 0 || C % G != 0)
        return AZ_ERR_BAD_ARG;
    if (H * W >= (1ll << 31) / 4 || B > 65535 || C > 65535 || H > 65535) return AZ_ERR_BAD_ARG;
    if (!gL && !gR) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == AZ_DTYPE_BF16) {
        using T = __nv_bfloat16;
        return gwc_bwd(static_cast<const T*>(gvol), static_cast<const T*>(L), static_cast<const T*>(R), static_cast<T*>(gL),
                       static_cast<T*>(gR), B, C, H, W, Dq, G, st);
    }
    using T = __half;
    return gwc_bwd(static_cast<const T*>(gvol), static_cast<const T*>(L), static_cast<const T*>(R), static_cast<T*>(gL),
                   static_cast<T*>(gR), B, C, H, W, Dq, G, st);
}
