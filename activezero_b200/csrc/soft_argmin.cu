// Fused soft-argmin (softmax over D + disparity regression), forward and backward
// (SURVEY.md §8a rows a4/a5).
// Reference: /root/reference/nets/psmnet/psmnet.py:200-201, 204-205, 212-217 and
//            /root/reference/nets/psmnet/psmnet_submodule.py:80-89.
//
// cost is [B,D,H,W] with D the slowest in-image axis (stride H*W), so the reduction over D is
// a per-thread serial loop over planes while a warp reads 512 contiguous bytes of one plane per
// request (128-bit loads, 8 planes in flight per thread).  One pass over the logits: online
// softmax in chunks of 8 planes -- chunk max, one rescale per chunk (skipped when the running
// max does not move), tree-summed chunk, running sums kept in double so the result stays well
// inside the 1e-4 px gate for flat distributions.  The forward also emits the log-sum-exp so
// the backward is a single read-modify-write pass with no second reduction.
#include <type_traits>

#include "common.cuh"

namespace az {

constexpr int kSAThreads = 256;
constexpr int kChunk = 8;
constexpr int kBwdDGroup = 16;  // planes per backward CTA (multiple of kChunk)
constexpr float kLog2e = 1.4426950408889634f;

template <int V> struct Vec;
template <> struct Vec<4> {
    using T = float4;
    static __device__ __forceinline__ void unpack(const float4& v, float* f) { f[0] = v.x; f[1] = v.y; f[2] = v.z; f[3] = v.w; }
    static __device__ __forceinline__ float4 pack(const float* f) { return make_float4(f[0], f[1], f[2], f[3]); }
};
template <> struct Vec<1> {
    using T = float;
    static __device__ __forceinline__ void unpack(const float& v, float* f) { f[0] = v; }
    static __device__ __forceinline__ float pack(const float* f) { return f[0]; }
};

// ---- 16-bit logits (bf16 / fp16): widened exactly after the load, gradients rounded once (RNE) at the store -------
template <typename T> struct Bits16;
template <> struct Bits16<__nv_bfloat16> {
    static __device__ __forceinline__ float widen(unsigned u) { return __uint_as_float(u << 16); }  // u: low 16 bits
    static __device__ __forceinline__ unsigned narrow(float f) { return __bfloat16_as_ushort(__float2bfloat16_rn(f)); }
};
template <> struct Bits16<__half> {
    static __device__ __forceinline__ float widen(unsigned u) { return __half2float(__ushort_as_half((unsigned short)u)); }
    static __device__ __forceinline__ unsigned narrow(float f) { return __half_as_ushort(__float2half_rn(f)); }
};

template <int V>
__device__ __forceinline__ void st_vec(float* p, const float* f) {
    st_stream(reinterpret_cast<typename Vec<V>::T*>(p), Vec<V>::pack(f));
}
template <int V, typename T>
__device__ __forceinline__ void st_vec(T* p, const float* f) {  // V = 4 / 8: p 8- / 16-byte aligned
    unsigned short* q = reinterpret_cast<unsigned short*>(p);
    if constexpr (V == 8) {
        unsigned w[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) w[i] = Bits16<T>::narrow(f[2 * i]) | (Bits16<T>::narrow(f[2 * i + 1]) << 16);
        __stcs(reinterpret_cast<uint4*>(q), make_uint4(w[0], w[1], w[2], w[3]));
    } else if (V == 4) {
        __stcs(reinterpret_cast<uint2*>(q), make_uint2(Bits16<T>::narrow(f[0]) | (Bits16<T>::narrow(f[1]) << 16),
                                                       Bits16<T>::narrow(f[2]) | (Bits16<T>::narrow(f[3]) << 16)));
    } else {
#pragma unroll
        for (int j = 0; j < V; ++j) __stcs(q + j, (unsigned short)Bits16<T>::narrow(f[j]));
    }
}
// V adjacent logits as loaded (raw), widened to fp32 where they are used: a 16-bit pass keeps its planes in flight as
// 16-bit words (half the registers of widened values).  Used where the pointer is aligned for the V-wide access.
template <typename T, int V> struct Lanes {
    using R = typename std::conditional<V == 8, uint4, typename std::conditional<V == 4, uint2, unsigned short>::type>::type;
    static __device__ __forceinline__ R ld(const T* p) { return __ldcs(reinterpret_cast<const R*>(p)); }
    static __device__ __forceinline__ void widen(const R& r, float* f) {
        if constexpr (V == 8) {
            const unsigned w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                f[2 * i] = Bits16<T>::widen(w[i] & 0xffffu);
                f[2 * i + 1] = Bits16<T>::widen(w[i] >> 16);
            }
        } else if constexpr (V == 4) {
            f[0] = Bits16<T>::widen(r.x & 0xffffu);
            f[1] = Bits16<T>::widen(r.x >> 16);
            f[2] = Bits16<T>::widen(r.y & 0xffffu);
            f[3] = Bits16<T>::widen(r.y >> 16);
        } else {
            f[0] = Bits16<T>::widen(r);
        }
    }
};
template <int V> struct Lanes<float, V> {
    using R = typename Vec<V>::T;
    static __device__ __forceinline__ R ld(const float* p) { return ld_stream(reinterpret_cast<const R*>(p)); }
    static __device__ __forceinline__ void widen(const R& r, float* f) { Vec<V>::unpack(r, f); }
};
// Four logits as raw words for the packed forward: ALIGNED = one 8-byte access, else four 2-byte ones (same bits).
template <bool ALIGNED>
__device__ __forceinline__ float4 ld_raw4(const float* p) { return ld_stream(reinterpret_cast<const float4*>(p)); }
template <bool ALIGNED, typename T>
__device__ __forceinline__ uint2 ld_raw4(const T* p) {
    if (ALIGNED) return __ldcs(reinterpret_cast<const uint2*>(p));
    const unsigned short* q = reinterpret_cast<const unsigned short*>(p);
    return make_uint2(__ldcs(q) | ((unsigned)__ldcs(q + 1) << 16), __ldcs(q + 2) | ((unsigned)__ldcs(q + 3) << 16));
}
// four -inf logits (planes past D) as raw words
template <typename T> __device__ __forceinline__ typename Lanes<T, 4>::R neg_inf4();
template <> __device__ __forceinline__ float4 neg_inf4<float>() { return make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY); }
template <> __device__ __forceinline__ uint2 neg_inf4<__nv_bfloat16>() { return make_uint2(0xff80ff80u, 0xff80ff80u); }
template <> __device__ __forceinline__ uint2 neg_inf4<__half>() { return make_uint2(0xfc00fc00u, 0xfc00fc00u); }
// Chunks of 8 planes loaded per pass by a thread of V pixels.  A 16-bit thread with 4 pixels loads two (16 planes x 8 B),
// one with 8 pixels one (8 planes x 16 B): either way its bytes per pass match the fp32 kernel's 8 planes x 16 B (what
// reaches the read-only ceiling, DESIGN.md §4.3).  The arithmetic is unchanged.
template <typename T, int V> constexpr int kFlight = (sizeof(T) == 4 || V == 8) ? 1 : 2;

// One thread owns V adjacent pixels.  n_vec = B*H*W/V work items; plane = H*W (floats).
template <typename T, int V>
__global__ void __launch_bounds__(kSAThreads) soft_argmin_fwd_kernel(const T* __restrict__ cost,
                                                                    float* __restrict__ disp,
                                                                    float* __restrict__ lse, int D,
                                                                    int64_t plane, int64_t n_vec) {
    using VT = typename Vec<V>::T;
    const int64_t t = (int64_t)blockIdx.x * kSAThreads + threadIdx.x;
    if (t >= n_vec) return;
    const int64_t pix = t * V;
    const int64_t b = pix / plane, hw = pix - b * plane;
    const T* src = cost + b * D * plane + hw;

    // m = running max.  Exponents are formed as (x - m) * log2e: the subtraction is exact for the
    // entries that carry weight (x close to m), so accuracy does not depend on the magnitude of the
    // logits, and every rounding (term exponent, rescale exponent) is relative to a SMALL number, which
    // keeps old and new partial sums consistent across rescales.
    float m[V];
    double s[V], ws[V];
#pragma unroll
    for (int j = 0; j < V; ++j) { m[j] = -INFINITY; s[j] = 0.0; ws[j] = 0.0; }

    for (int d0 = 0; d0 < D; d0 += kChunk) {
        float x[kChunk][V];
#pragma unroll
        for (int k = 0; k < kChunk; ++k) {
            if (d0 + k < D) {
                Lanes<T, V>::widen(Lanes<T, V>::ld(src + (int64_t)(d0 + k) * plane), x[k]);
            } else {
#pragma unroll
                for (int j = 0; j < V; ++j) x[k][j] = -INFINITY;
            }
        }
#pragma unroll
        for (int j = 0; j < V; ++j) {
            float cm = x[0][j];
#pragma unroll
            for (int k = 1; k < kChunk; ++k) cm = fmaxf(cm, x[k][j]);
            if (cm > m[j]) {  // rescale the running sums (exp2(-inf) = 0 on the first chunk)
                const double sc = (double)fast_ex2((m[j] - cm) * kLog2e);
                s[j] *= sc;
                ws[j] *= sc;
                m[j] = cm;
            }
            const float ref = (m[j] == -INFINITY) ? 0.f : m[j];  // leading -inf planes contribute 0
            float e[kChunk];
#pragma unroll
            for (int k = 0; k < kChunk; ++k) e[k] = fast_ex2((x[k][j] - ref) * kLog2e);
            // tree sums of the chunk in fp32, running sums in fp64
            const float s01 = e[0] + e[1], s23 = e[2] + e[3], s45 = e[4] + e[5], s67 = e[6] + e[7];
            const float w01 = e[1], w23 = fmaf(e[3], 3.f, e[2] * 2.f);
            const float w45 = fmaf(e[5], 5.f, e[4] * 4.f), w67 = fmaf(e[7], 7.f, e[6] * 6.f);
            const float cs = (s01 + s23) + (s45 + s67);
            const float cw = (w01 + w23) + (w45 + w67);  // sum_k k*e[k], k local
            s[j] += (double)cs;
            ws[j] += (double)cw + (double)d0 * (double)cs;
        }
    }
    float o[V], l[V];
#pragma unroll
    for (int j = 0; j < V; ++j) o[j] = (float)(ws[j] / s[j]);
    *reinterpret_cast<VT*>(disp + pix) = Vec<V>::pack(o);
    if (lse != nullptr) {
        // saved for the backward: plane 0 = max logit m, plane 1 = log2(sum_d 2^((x_d - m)*log2e));
        // the backward forms p_d = 2^((x_d - m)*log2e - plane1) with the same exact subtraction.
        const int64_t total = n_vec * V;
        *reinterpret_cast<VT*>(lse + pix) = Vec<V>::pack(m);
#pragma unroll
        for (int j = 0; j < V; ++j) l[j] = log2f((float)s[j]);
        *reinterpret_cast<VT*>(lse + total + pix) = Vec<V>::pack(l);
    }
}


// ------------------------------------------------------------------------------------------
// Forward, packed form (what az_soft_argmin_fwd launches for the vector path).  Same algorithm as the
// generic kernel above -- online softmax in chunks of 8 planes, exponents formed from the exact
// difference to the running max -- with the arithmetic re-balanced for the B200 issue/XU budget
// (round-1 ncu: XU pipe 60 %, issue 44 %, 0.89 of the read-only ceiling):
//   * the subtract / scale / tree-sum / weighted-sum of two adjacent pixels run as ONE packed
//     fp32x2 instruction (sub/mul/add/fma.rn.f32x2 -> FADD2/FMUL2/FFMA2): ~5 instead of ~7 issue slots
//     per logit;
//   * BITS: the float->double conversions of the chunk sums (XU pipe, next to the ex2) are done with
//     integer shifts instead (an fp32 Kahan / TwoSum accumulation was emulated and rejected: the
//     rescale products and the d0*cs term need error-free transforms to stay at the fp64 sums'
//     2e-5 px, which costs more issue slots than it saves);
//   * POLY > 0: the last POLY of the 8 exponentials of a chunk are evaluated on the FMA pipe
//     (Cody-Waite split + degree-6 polynomial, packed) instead of MUFU.
// ------------------------------------------------------------------------------------------
typedef unsigned long long u64p;
__device__ __forceinline__ u64p pk(float lo, float hi) { u64p r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void upk(u64p v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ u64p padd(u64p a, u64p b) { u64p r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ u64p psub(u64p a, u64p b) { u64p r; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ u64p pmul(u64p a, u64p b) { u64p r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ u64p pfma(u64p a, u64p b, u64p c) { u64p r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }

// 2^t for a packed pair, t <= 0, on the FMA/ALU pipes: t = n + f, n = rint(t), |f| <= 1/2,
// 2^f = degree-6 Taylor polynomial in f*ln2 (truncation 1.2e-7 relative), scaled by 2^n through the
// exponent field.  t is clamped at -126 (a term below 2^-126 of the maximum carries no weight).
__device__ __forceinline__ u64p pexp2_poly(u64p t) {
    float t0, t1;
    upk(t, t0, t1);
    t0 = fmaxf(t0, -126.0f);
    t1 = fmaxf(t1, -126.0f);
    const float kMagic = 12582912.0f;  // 1.5 * 2^23: adding it rounds to the nearest integer
    const float r0 = __fadd_rn(t0, kMagic), r1 = __fadd_rn(t1, kMagic);
    const u64p n = psub(pk(r0, r1), pk(kMagic, kMagic));
    const u64p f = psub(pk(t0, t1), n);
    // coefficients ln2^k / k!
    u64p p = pk(1.5403530393381608e-4f, 1.5403530393381608e-4f);
    p = pfma(p, f, pk(1.3333558146428443e-3f, 1.3333558146428443e-3f));
    p = pfma(p, f, pk(9.6181291076284772e-3f, 9.6181291076284772e-3f));
    p = pfma(p, f, pk(5.5504108664821580e-2f, 5.5504108664821580e-2f));
    p = pfma(p, f, pk(2.4022650695910072e-1f, 2.4022650695910072e-1f));
    p = pfma(p, f, pk(6.9314718055994531e-1f, 6.9314718055994531e-1f));
    p = pfma(p, f, pk(1.0f, 1.0f));
    float p0, p1;
    upk(p, p0, p1);
    // r = kMagic + n exactly, so its low mantissa bits hold n (two's complement): shift them into the exponent
    p0 = __int_as_float(__float_as_int(p0) + (__float_as_int(r0) << 23));
    p1 = __int_as_float(__float_as_int(p1) + (__float_as_int(r1) << 23));
    return pk(p0, p1);
}

// float -> double for a non-negative, normal-or-zero float with integer instructions (exact for
// normals; +0 maps to 2^-127, which no sum notices): the F2F.F64.F32 conversion runs on the XU pipe
// next to the exponentials that bound this kernel.
template <bool BITS>
__device__ __forceinline__ double to_double_pos(float f) {
    if (BITS) {
        const unsigned u = __float_as_uint(f);
        return __hiloint2double((int)((u >> 3) + 0x38000000u), (int)(u << 29));
    }
    return (double)f;
}

// T = float: one chunk of 8 planes per pass.  T = bf16 / fp16 (logits widened at the load): two chunks per pass, each
// reduced exactly as the fp32 kernel reduces it; ALIGNED = false takes 2-byte loads and 4-byte stores (a view with
// a storage offset) with the same arithmetic.
template <typename T, int POLY, bool BITS, bool ALIGNED = true>
__global__ void __launch_bounds__(kSAThreads) soft_argmin_fwd_packed_kernel(const T* __restrict__ cost,
                                                                           float* __restrict__ disp,
                                                                           float* __restrict__ lse, int D,
                                                                           int64_t plane, int64_t n_vec) {
    constexpr int NF = kFlight<T, 4>;
    const int64_t t = (int64_t)blockIdx.x * kSAThreads + threadIdx.x;
    if (t >= n_vec) return;
    const int64_t pix = t * 4;
    const int64_t b = pix / plane, hw = pix - b * plane;
    const T* src = cost + b * D * plane + hw;
    const u64p kL2 = pk(kLog2e, kLog2e);

    float m[4];
    double s[4], ws[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) { m[j] = -INFINITY; s[j] = 0.0; ws[j] = 0.0; }

    for (int d00 = 0; d00 < D; d00 += NF * kChunk) {
        typename Lanes<T, 4>::R v[NF * kChunk];  // 16-bit: raw words until use (registers for all 16 planes in flight)
#pragma unroll
        for (int k = 0; k < NF * kChunk; ++k) {
            if (d00 + k < D) v[k] = ld_raw4<ALIGNED>(src + (int64_t)(d00 + k) * plane);
            else v[k] = neg_inf4<T>();
        }
#pragma unroll
        for (int c = 0; c < NF; ++c) {
        const int d0 = d00 + c * kChunk;
        if (c > 0 && d0 >= D) break;  // (uniform) a pass may end in a chunk past the last plane
        const double dd0 = (double)d0;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            float xa[kChunk], xb[kChunk];
#pragma unroll
            for (int k = 0; k < kChunk; ++k) {
                float f[4];
                Lanes<T, 4>::widen(v[c * kChunk + k], f);
                xa[k] = f[2 * h];
                xb[k] = f[2 * h + 1];
            }
            float ca = xa[0], cb = xb[0];
#pragma unroll
            for (int k = 1; k < kChunk; ++k) { ca = fmaxf(ca, xa[k]); cb = fmaxf(cb, xb[k]); }
            float& ma = m[2 * h];
            float& mb = m[2 * h + 1];
            if (ca > ma) {  // rescale the running sums (exp2(-inf) = 0 on the first chunk)
                const double r = (double)fast_ex2((ma - ca) * kLog2e);
                s[2 * h] *= r;
                ws[2 * h] *= r;
                ma = ca;
            }
            if (cb > mb) {
                const double r = (double)fast_ex2((mb - cb) * kLog2e);
                s[2 * h + 1] *= r;
                ws[2 * h + 1] *= r;
                mb = cb;
            }
            const u64p ref = pk(ma == -INFINITY ? 0.f : ma, mb == -INFINITY ? 0.f : mb);  // leading -inf planes contribute 0
            u64p e[kChunk];
#pragma unroll
            for (int k = 0; k < kChunk; ++k) {
                const u64p a = pmul(psub(pk(xa[k], xb[k]), ref), kL2);
                if (k >= kChunk - POLY) {
                    e[k] = pexp2_poly(a);
                } else {
                    float a0, a1;
                    upk(a, a0, a1);
                    e[k] = pk(fast_ex2(a0), fast_ex2(a1));
                }
            }
            // tree sums of the chunk in (packed) fp32, running sums in fp64
            const u64p s01 = padd(e[0], e[1]), s23 = padd(e[2], e[3]), s45 = padd(e[4], e[5]), s67 = padd(e[6], e[7]);
            const u64p cs = padd(padd(s01, s23), padd(s45, s67));
            const u64p w23 = pfma(e[3], pk(3.f, 3.f), padd(e[2], e[2]));
            const u64p w45 = pfma(e[5], pk(5.f, 5.f), pmul(e[4], pk(4.f, 4.f)));
            const u64p w67 = pfma(e[7], pk(7.f, 7.f), pmul(e[6], pk(6.f, 6.f)));
            const u64p cw = padd(padd(e[1], w23), padd(w45, w67));  // sum_k k*e[k], k local
            float csa, csb, cwa, cwb;
            upk(cs, csa, csb);
            upk(cw, cwa, cwb);
            const double dsa = to_double_pos<BITS>(csa), dsb = to_double_pos<BITS>(csb);
            s[2 * h] += dsa;
            s[2 * h + 1] += dsb;
            ws[2 * h] += fma(dd0, dsa, to_double_pos<BITS>(cwa));
            ws[2 * h + 1] += fma(dd0, dsb, to_double_pos<BITS>(cwb));
        }
        }
    }
    float o[4], l[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        o[j] = (float)(ws[j] / s[j]);
        l[j] = log2f((float)s[j]);
    }
    const int64_t total = n_vec * 4;
    if (ALIGNED) {
        *reinterpret_cast<float4*>(disp + pix) = make_float4(o[0], o[1], o[2], o[3]);
        if (lse != nullptr) {
            *reinterpret_cast<float4*>(lse + pix) = make_float4(m[0], m[1], m[2], m[3]);
            *reinterpret_cast<float4*>(lse + total + pix) = make_float4(l[0], l[1], l[2], l[3]);
        }
    } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            disp[pix + j] = o[j];
            if (lse != nullptr) {
                lse[pix + j] = m[j];
                lse[total + pix + j] = l[j];
            }
        }
    }
}

// T = bf16 / fp16: the gradient is formed in fp32 exactly as for fp32 logits and rounded once (RNE) at the store.
// V = 8 (8 pixels, 16-byte accesses, 8 planes per pass) where H*W % 8 == 0 and the pointers allow it, else V = 4 with
// the CTA's 16 planes loaded at once: both keep the fp32 kernel's bytes per pass; V = 8 measured faster (§4.12).
template <typename T, int V, int KF = kFlight<T, V> * kChunk>
__global__ void __launch_bounds__(kSAThreads) soft_argmin_bwd_kernel(const T* __restrict__ cost,
                                                                    const float* __restrict__ disp,
                                                                    const float* __restrict__ lse,
                                                                    const float* __restrict__ gdisp,
                                                                    T* __restrict__ gcost, int D,
                                                                    int64_t plane, int64_t n_vec, int dgroup) {
    // grid.y splits the D planes into groups of `dgroup`: short-lived CTAs keep the store half of this
    // read-modify-write stream nearer the write-only ceiling (benchmarks/micro/store_patterns.cu)
    constexpr int VW = V == 8 ? 4 : V;  // fp32 vector width of the disp / lse / gdisp reads
    using VT = typename Vec<VW>::T;
    const int64_t t = (int64_t)blockIdx.x * kSAThreads + threadIdx.x;
    if (t >= n_vec) return;
    const int64_t pix = t * V;
    const int64_t b = pix / plane, hw = pix - b * plane;
    const T* src = cost + b * D * plane + hw;
    T* dst = gcost + b * D * plane + hw;
    const int dbeg = blockIdx.y * dgroup, dend = min(D, dbeg + dgroup);
    float o[V], mx[V], lb[V], g[V];
#pragma unroll
    for (int q = 0; q < V; q += VW) {
        Vec<VW>::unpack(*reinterpret_cast<const VT*>(disp + pix + q), o + q);
        Vec<VW>::unpack(*reinterpret_cast<const VT*>(lse + pix + q), mx + q);
        Vec<VW>::unpack(*reinterpret_cast<const VT*>(lse + n_vec * V + pix + q), lb + q);
        Vec<VW>::unpack(*reinterpret_cast<const VT*>(gdisp + pix + q), g + q);
    }
    for (int d0 = dbeg; d0 < dend; d0 += KF) {
        typename Lanes<T, V>::R v[KF];
#pragma unroll
        for (int k = 0; k < KF; ++k)
            if (d0 + k < dend) v[k] = Lanes<T, V>::ld(src + (int64_t)(d0 + k) * plane);
#pragma unroll
        for (int k = 0; k < KF; ++k) {
            if (d0 + k < dend) {
                float x[V], r[V];
                Lanes<T, V>::widen(v[k], x);
                const float dd = (float)(d0 + k);
#pragma unroll
                for (int j = 0; j < V; ++j) {
                    const float p = fast_ex2(fmaf(x[j] - mx[j], kLog2e, -lb[j]));
                    r[j] = p * (dd - o[j]) * g[j];
                }
                st_vec<V>(dst + (int64_t)(d0 + k) * plane, r);
            }
        }
    }
}

}  // namespace az

using namespace az;

extern "C" int az_soft_argmin_fwd(const float* cost, float* disp, float* lse, int64_t B, int64_t D, int64_t H,
                                  int64_t W, void* stream) {
    if (!cost || !disp || B <= 0 || D <= 0 || H <= 0 || W <= 0) return AZ_ERR_BAD_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t plane = H * W, total = B * plane;
    const bool vec = (plane % 4 == 0) && aligned16(cost) && aligned16(disp) && (lse == nullptr || aligned16(lse));
    if (vec) {
        const int64_t n = total / 4;
        const unsigned grid = (unsigned)ceil_div(n, kSAThreads);
        // 0 = generic kernel; 1 = packed; 2 = packed + integer conversions; 3 / 4 = (2) + 2 / 4 polynomial exp2 per chunk
        switch (az::tuning("AZ_SA_FWD", 2)) {
            case 0: soft_argmin_fwd_kernel<float, 4><<<grid, kSAThreads, 0, st>>>(cost, disp, lse, (int)D, plane, n); break;
            case 1: soft_argmin_fwd_packed_kernel<float, 0, false><<<grid, kSAThreads, 0, st>>>(cost, disp, lse, (int)D, plane, n); break;
            case 3: soft_argmin_fwd_packed_kernel<float, 2, true><<<grid, kSAThreads, 0, st>>>(cost, disp, lse, (int)D, plane, n); break;
            case 4: soft_argmin_fwd_packed_kernel<float, 4, true><<<grid, kSAThreads, 0, st>>>(cost, disp, lse, (int)D, plane, n); break;
            default: soft_argmin_fwd_packed_kernel<float, 0, true><<<grid, kSAThreads, 0, st>>>(cost, disp, lse, (int)D, plane, n); break;
        }
    } else {
        soft_argmin_fwd_kernel<float, 1><<<(unsigned)ceil_div(total, kSAThreads), kSAThreads, 0, st>>>(
            cost, disp, lse, (int)D, plane, total);
    }
    AZ_LAUNCH_CHECK();
    return 0;
}

extern "C" int az_soft_argmin_bwd(const float* cost, const float* disp, const float* lse, const float* gdisp,
                                  float* gcost, int64_t B, int64_t D, int64_t H, int64_t W, void* stream) {
    if (!cost || !disp || !lse || !gdisp || !gcost || B <= 0 || D <= 0 || H <= 0 || W <= 0) return AZ_ERR_BAD_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t plane = H * W, total = B * plane;
    const bool vec = (plane % 4 == 0) && aligned16(cost) && aligned16(disp) && aligned16(lse) && aligned16(gdisp) &&
                     aligned16(gcost);
    const int dgroup = kBwdDGroup;
    const unsigned ngroups = (unsigned)ceil_div(D, dgroup);
    if (ngroups > 65535) return AZ_ERR_BAD_ARG;
    if (vec) {
        const int64_t n = total / 4;
        dim3 grid((unsigned)ceil_div(n, kSAThreads), ngroups);
        soft_argmin_bwd_kernel<float, 4><<<grid, kSAThreads, 0, st>>>(cost, disp, lse, gdisp, gcost, (int)D, plane, n, dgroup);
    } else {
        dim3 grid((unsigned)ceil_div(total, kSAThreads), ngroups);
        soft_argmin_bwd_kernel<float, 1><<<grid, kSAThreads, 0, st>>>(cost, disp, lse, gdisp, gcost, (int)D, plane, total,
                                                                      dgroup);
    }
    AZ_LAUNCH_CHECK();
    return 0;
}

// 16-bit logits.  The forward picks its arithmetic by the fp32 operator's shape rule alone (the packed kernel when
// H*W % 4 == 0, else the generic one), never by the alignment of the 16-bit pointer, so that it matches the fp32
// operator on cost.float() (a fresh, aligned tensor) for any view; the AZ_SA_FWD knob is not consulted.  The backward's
// arithmetic is the same per element at every vector width, so its width follows the shape and the pointers.
template <typename T>
static int soft_argmin_fwd16(const T* cost, float* disp, float* lse, int64_t B, int64_t D, int64_t H, int64_t W,
                             cudaStream_t st) {
    const int64_t plane = H * W, total = B * plane;
    if (plane % 4 == 0) {
        const int64_t n = total / 4;
        const unsigned grid = (unsigned)ceil_div(n, kSAThreads);
        const bool al = ((reinterpret_cast<uintptr_t>(cost) & 7u) == 0) && aligned16(disp) &&
                        (lse == nullptr || aligned16(lse));
        if (al) soft_argmin_fwd_packed_kernel<T, 0, true, true><<<grid, kSAThreads, 0, st>>>(cost, disp, lse, (int)D, plane, n);
        else soft_argmin_fwd_packed_kernel<T, 0, true, false><<<grid, kSAThreads, 0, st>>>(cost, disp, lse, (int)D, plane, n);
    } else {
        soft_argmin_fwd_kernel<T, 1><<<(unsigned)ceil_div(total, kSAThreads), kSAThreads, 0, st>>>(cost, disp, lse,
                                                                                                  (int)D, plane, total);
    }
    AZ_LAUNCH_CHECK();
    return 0;
}

template <typename T>
static int soft_argmin_bwd16(const T* cost, const float* disp, const float* lse, const float* gdisp, T* gcost,
                             int64_t B, int64_t D, int64_t H, int64_t W, cudaStream_t st) {
    const int64_t plane = H * W, total = B * plane;
    const bool vec = (plane % 4 == 0) && ((reinterpret_cast<uintptr_t>(cost) & 7u) == 0) &&
                     ((reinterpret_cast<uintptr_t>(gcost) & 7u) == 0) && aligned16(disp) && aligned16(lse) &&
                     aligned16(gdisp);
    const int dgroup = kBwdDGroup;
    const unsigned ngroups = (unsigned)ceil_div(D, dgroup);
    if (ngroups > 65535) return AZ_ERR_BAD_ARG;
    if (vec && plane % 8 == 0 && aligned16(cost) && aligned16(gcost)) {
        const int64_t n = total / 8;
        dim3 grid((unsigned)ceil_div(n, kSAThreads), ngroups);
        soft_argmin_bwd_kernel<T, 8><<<grid, kSAThreads, 0, st>>>(cost, disp, lse, gdisp, gcost, (int)D, plane, n, dgroup);
    } else if (vec) {
        const int64_t n = total / 4;
        dim3 grid((unsigned)ceil_div(n, kSAThreads), ngroups);
        soft_argmin_bwd_kernel<T, 4><<<grid, kSAThreads, 0, st>>>(cost, disp, lse, gdisp, gcost, (int)D, plane, n, dgroup);
    } else {
        dim3 grid((unsigned)ceil_div(total, kSAThreads), ngroups);
        soft_argmin_bwd_kernel<T, 1><<<grid, kSAThreads, 0, st>>>(cost, disp, lse, gdisp, gcost, (int)D, plane, total,
                                                                  dgroup);
    }
    AZ_LAUNCH_CHECK();
    return 0;
}

extern "C" int az_soft_argmin_fwd_16(const void* cost, float* disp, float* lse, int64_t B, int64_t D, int64_t H,
                                     int64_t W, int dtype, void* stream) {
    if (!cost || !disp || B <= 0 || D <= 0 || H <= 0 || W <= 0) return AZ_ERR_BAD_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == AZ_DTYPE_BF16)
        return soft_argmin_fwd16(static_cast<const __nv_bfloat16*>(cost), disp, lse, B, D, H, W, st);
    if (dtype == AZ_DTYPE_F16) return soft_argmin_fwd16(static_cast<const __half*>(cost), disp, lse, B, D, H, W, st);
    return AZ_ERR_BAD_ARG;
}

extern "C" int az_soft_argmin_bwd_16(const void* cost, const float* disp, const float* lse, const float* gdisp,
                                     void* gcost, int64_t B, int64_t D, int64_t H, int64_t W, int dtype, void* stream) {
    if (!cost || !disp || !lse || !gdisp || !gcost || B <= 0 || D <= 0 || H <= 0 || W <= 0) return AZ_ERR_BAD_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == AZ_DTYPE_BF16)
        return soft_argmin_bwd16(static_cast<const __nv_bfloat16*>(cost), disp, lse, gdisp,
                                 static_cast<__nv_bfloat16*>(gcost), B, D, H, W, st);
    if (dtype == AZ_DTYPE_F16)
        return soft_argmin_bwd16(static_cast<const __half*>(cost), disp, lse, gdisp, static_cast<__half*>(gcost), B, D,
                                 H, W, st);
    return AZ_ERR_BAD_ARG;
}
