// Trilinear upsample fused into soft-argmin (SURVEY.md §8f rank 1, a "next" row).
// Reference: /root/reference/nets/psmnet/psmnet.py:186-197, 208-211
//   cost = F.interpolate(cost, (maxdisp, 4H, 4W), mode="trilinear", align_corners=False)
// followed by :200-201 / :212-217 softmax + DisparityRegression.  The reference materialises the
// [B,D,4H,4W] logits (401 MB per pair at 544x960, D=192) only for the soft-argmin to read them
// back; here the kernel reads the [B,Dq,Hq,Wq] low-resolution logits (6.3 MB per pair), rebuilds
// each full-resolution logit on the fly and reduces it immediately -- ~60x less HBM traffic, so
// the op becomes MUFU-bound (one ex2 per full-resolution logit).
//
// Interpolation follows torch's upsample_trilinear3d with align_corners=False:
//   src = max(scale*(dst+0.5)-0.5, 0), scale = in/out (float); i0 = int(src); i1 = i0 + (i0 < in-1);
//   l1 = src - i0; l0 = 1 - l1.
// It is separable: v_q(y,x) = bilinear_hw(lowres[q]) once per low-res plane, then
// logit_d = l0(d)*v_{q0(d)} + l1(d)*v_{q1(d)}.
//
// Backward, deterministic (torch's own trilinear backward uses float atomics):
//   1. per output pixel, G[q] = sum_d w(d,q) * p_d*(d-disp)*g      -> workspace [B,Dq,H,W]
//   2. reduce along x with the horizontal interpolation weights     -> workspace [B,Dq,H,Wq]
//   3. reduce along y with the vertical weights                     -> glow [B,Dq,Hq,Wq]
#include "common.cuh"

namespace az {

constexpr float kLog2eU = 1.4426950408889634f;
constexpr int kUTW = 32, kUTH = 8;  // output tile of one CTA

struct Lerp {
    int i0, i1;
    float l0, l1;
};

__device__ __forceinline__ Lerp src_index(float scale, int dst, int in_size) {
    float src = scale * ((float)dst + 0.5f) - 0.5f;
    src = src < 0.f ? 0.f : src;
    Lerp r;
    r.i0 = min((int)src, in_size - 1);
    r.i1 = r.i0 + (r.i0 < in_size - 1 ? 1 : 0);
    r.l1 = src - (float)r.i0;
    r.l0 = 1.0f - r.l1;
    return r;
}

// Shared-memory tile of the low-res logits under one output tile, and the per-thread bilinear taps.
struct Taps {
    int o00, o01, o10, o11;
    float w00, w01, w10, w11;
};

__device__ __forceinline__ float bil(const float* __restrict__ plane, const Taps& t) {
    // torch's nesting: h0*(w0*a + w1*b) + h1*(w0*c + w1*d), folded into four products
    return fmaf(t.w11, plane[t.o11], fmaf(t.w10, plane[t.o10], fmaf(t.w01, plane[t.o01], t.w00 * plane[t.o00])));
}

// Loads the [Dq][fh][fw] footprint of this CTA's output tile.  64 threads walk the fh*fw positions (one
// integer division each), the 4 groups of 64 interleave over the Dq planes: no div/mod in the inner loop.  16-bit
// logits are widened (exactly) here: the tile is fp32 for every input type.
template <typename T>
__device__ __forceinline__ void load_tile(const T* __restrict__ low, float* __restrict__ tile, int b, int Dq, int Hq,
                                          int Wq, int h_lo, int w_lo, int fh, int fw, int FHW) {
    const int tid = threadIdx.y * kUTW + threadIdx.x;
    const int npos = fh * fw;
    const size_t plane = (size_t)Hq * Wq;
    for (int pos = tid & 63; pos < npos; pos += 64) {
        const int hh = pos / fw, ww = pos - hh * fw;
        const T* src = low + (size_t)b * Dq * plane + (size_t)(h_lo + hh) * Wq + (w_lo + ww);
        for (int q = tid >> 6; q < Dq; q += (kUTW * kUTH) >> 6) tile[q * FHW + pos] = ld_f32(src + (size_t)q * plane);
    }
}

// Depth look-up tables shared by the CTA: l1[d] = weight of plane q1(d); dstart[q] = first d whose
// lower plane is q (dstart[Dq] = D).  Upsampling => q0(d) is non-decreasing with steps <= 1, so the
// d axis splits into Dq consecutive intervals, on each of which the logit is a monotone lerp
// between v_q and v_{q1} -- its maximum is attained at the interval's first or last sample.
__device__ __forceinline__ void build_depth_lut(float* __restrict__ l1, int* __restrict__ dstart, float sd, int Dq, int D) {
    const int tid = threadIdx.y * kUTW + threadIdx.x;
    for (int d = tid; d < D; d += kUTW * kUTH) {
        const Lerp ld = src_index(sd, d, Dq);
        l1[d] = ld.l1;
        if (d == 0 || src_index(sd, d - 1, Dq).i0 != ld.i0) dstart[ld.i0] = d;
    }
    if (tid == 0) dstart[Dq] = D;
}

// grid = (ceil(W/32), ceil(H/8), B), block = (32, 8)
// smem: tile[Dq*FHW] floats | l1[D] floats | dstart[Dq+1] ints
template <typename T>
__global__ void __launch_bounds__(kUTW * kUTH) upsample_soft_argmin_fwd_kernel(
    const T* __restrict__ low, float* __restrict__ disp, float* __restrict__ stats, int Dq, int Hq, int Wq, int D,
    int H, int W, float sd, float sh, float sw, int FHW, int64_t total) {
    extern __shared__ float tile[];
    float* l1 = tile + (size_t)Dq * FHW;
    int* dstart = reinterpret_cast<int*>(l1 + D);
    const int b = blockIdx.z;
    const int x0 = blockIdx.x * kUTW, y0 = blockIdx.y * kUTH;
    const int x1 = min(x0 + kUTW, W) - 1, y1 = min(y0 + kUTH, H) - 1;
    const int h_lo = src_index(sh, y0, Hq).i0, h_hi = src_index(sh, y1, Hq).i1;
    const int w_lo = src_index(sw, x0, Wq).i0, w_hi = src_index(sw, x1, Wq).i1;
    const int fh = h_hi - h_lo + 1, fw = w_hi - w_lo + 1;
    load_tile(low, tile, b, Dq, Hq, Wq, h_lo, w_lo, fh, fw, FHW);
    build_depth_lut(l1, dstart, sd, Dq, D);
    __syncthreads();
    const int x = x0 + threadIdx.x, y = y0 + threadIdx.y;
    if (x >= W || y >= H) return;
    const Lerp ly = src_index(sh, y, Hq), lx = src_index(sw, x, Wq);
    Taps t;
    t.o00 = (ly.i0 - h_lo) * fw + (lx.i0 - w_lo);
    t.o01 = (ly.i0 - h_lo) * fw + (lx.i1 - w_lo);
    t.o10 = (ly.i1 - h_lo) * fw + (lx.i0 - w_lo);
    t.o11 = (ly.i1 - h_lo) * fw + (lx.i1 - w_lo);
    t.w00 = ly.l0 * lx.l0; t.w01 = ly.l0 * lx.l1; t.w10 = ly.l1 * lx.l0; t.w11 = ly.l1 * lx.l1;

    // online softmax over the Dq depth intervals; interval sums in fp32, running sums in fp64
    float m = -INFINITY;
    double s = 0.0, ws = 0.0;
    float va = bil(tile, t);
    for (int q = 0; q < Dq; ++q) {
        const float vb = (q + 1 < Dq) ? bil(tile + (q + 1) * FHW, t) : va;
        const float diff = vb - va;
        const int db = dstart[q], de = dstart[q + 1];
        if (de > db) {
            const float lf = fmaf(l1[db], diff, va), ll = fmaf(l1[de - 1], diff, va);
            const float cm = fmaxf(lf, ll);
            if (cm > m) {
                const double sc = (double)fast_ex2((m - cm) * kLog2eU);
                s *= sc;
                ws *= sc;
                m = cm;
            }
            float cs = 0.f, cw = 0.f, kf = 0.f;
            for (int d = db; d < de; ++d) {
                const float e = fast_ex2((fmaf(l1[d], diff, va) - m) * kLog2eU);
                cs += e;
                cw = fmaf(kf, e, cw);
                kf += 1.0f;
            }
            s += (double)cs;
            ws += (double)cw + (double)db * (double)cs;
        }
        va = vb;
    }
    const size_t pix = ((size_t)b * H + y) * W + x;
    disp[pix] = (float)(ws / s);
    if (stats != nullptr) {
        stats[pix] = m;
        stats[total + pix] = log2f((float)s);
    }
}

// backward stage 1: per-pixel gradient w.r.t. the Dq interpolated planes v_q(y,x).  G: [B,Dq,H,W]
template <typename T>
__global__ void __launch_bounds__(kUTW * kUTH) upsample_soft_argmin_bwd_pix_kernel(
    const T* __restrict__ low, const float* __restrict__ disp, const float* __restrict__ stats,
    const float* __restrict__ gdisp, float* __restrict__ G, int Dq, int Hq, int Wq, int D, int H, int W, float sd,
    float sh, float sw, int FHW, int64_t total) {
    extern __shared__ float tile[];
    float* l1 = tile + (size_t)Dq * FHW;
    int* dstart = reinterpret_cast<int*>(l1 + D);
    const int b = blockIdx.z;
    const int x0 = blockIdx.x * kUTW, y0 = blockIdx.y * kUTH;
    const int x1 = min(x0 + kUTW, W) - 1, y1 = min(y0 + kUTH, H) - 1;
    const int h_lo = src_index(sh, y0, Hq).i0, h_hi = src_index(sh, y1, Hq).i1;
    const int w_lo = src_index(sw, x0, Wq).i0, w_hi = src_index(sw, x1, Wq).i1;
    const int fh = h_hi - h_lo + 1, fw = w_hi - w_lo + 1;
    load_tile(low, tile, b, Dq, Hq, Wq, h_lo, w_lo, fh, fw, FHW);
    build_depth_lut(l1, dstart, sd, Dq, D);
    __syncthreads();
    const int x = x0 + threadIdx.x, y = y0 + threadIdx.y;
    if (x >= W || y >= H) return;
    const Lerp ly = src_index(sh, y, Hq), lx = src_index(sw, x, Wq);
    Taps t;
    t.o00 = (ly.i0 - h_lo) * fw + (lx.i0 - w_lo);
    t.o01 = (ly.i0 - h_lo) * fw + (lx.i1 - w_lo);
    t.o10 = (ly.i1 - h_lo) * fw + (lx.i0 - w_lo);
    t.o11 = (ly.i1 - h_lo) * fw + (lx.i1 - w_lo);
    t.w00 = ly.l0 * lx.l0; t.w01 = ly.l0 * lx.l1; t.w10 = ly.l1 * lx.l0; t.w11 = ly.l1 * lx.l1;

    const size_t pix = ((size_t)b * H + y) * W + x;
    const float m = stats[pix], l2s = stats[total + pix], out = disp[pix], g = gdisp[pix];
    const size_t HW = (size_t)H * W;
    float* Gp = G + (size_t)b * Dq * HW + (size_t)y * W + x;
    float va = bil(tile, t);
    float carry = 0.f;  // gradient already collected for plane q as the UPPER plane of interval q-1
    for (int q = 0; q < Dq; ++q) {
        const bool top = q + 1 >= Dq;
        const float vb = top ? va : bil(tile + (q + 1) * FHW, t);
        const float diff = vb - va;
        const int db = dstart[q], de = dstart[q + 1];
        float ga = 0.f, gb = 0.f, df = (float)db;
        for (int d = db; d < de; ++d) {
            const float w1 = l1[d];
            const float p = fast_ex2(fmaf(fmaf(w1, diff, va) - m, kLog2eU, -l2s));
            const float gc = p * (df - out) * g;
            gb = fmaf(w1, gc, gb);
            ga += gc;
            df += 1.0f;
        }
        ga -= gb;  // sum (1 - w1) * gc
        Gp[(size_t)q * HW] = carry + (top ? ga + gb : ga);
        carry = gb;
        va = vb;
    }
}

// ------------------------------------------------------------------------------------------
// Depth scale exactly 4 (D == 4*Dq, the only case PSMNet uses: psmnet.py:186-211).  The depth
// weights are then the constants {1/8, 3/8, 5/8, 7/8} (exact in binary): interval q covers
// d = 4q+2 .. 4q+5; d = 0,1 clamp to plane 0 and d = D-2, D-1 clamp to plane Dq-1.  The four
// samples of an interval are unrolled with immediate weights -- no look-up tables, no inner
// loop: ~45 instructions and 4 ex2 per interval.
// ------------------------------------------------------------------------------------------
struct TileGeom {
    int h_lo, w_lo, fh, fw;
};

__device__ __forceinline__ TileGeom tile_geom(float sh, float sw, int Hq, int Wq, int H, int W) {
    const int x0 = blockIdx.x * kUTW, y0 = blockIdx.y * kUTH;
    const int x1 = min(x0 + kUTW, W) - 1, y1 = min(y0 + kUTH, H) - 1;
    TileGeom g;
    g.h_lo = src_index(sh, y0, Hq).i0;
    g.w_lo = src_index(sw, x0, Wq).i0;
    g.fh = src_index(sh, y1, Hq).i1 - g.h_lo + 1;
    g.fw = src_index(sw, x1, Wq).i1 - g.w_lo + 1;
    return g;
}

__device__ __forceinline__ Taps make_taps(float sh, float sw, int y, int x, int Hq, int Wq, const TileGeom& g) {
    const Lerp ly = src_index(sh, y, Hq), lx = src_index(sw, x, Wq);
    Taps t;
    t.o00 = (ly.i0 - g.h_lo) * g.fw + (lx.i0 - g.w_lo);
    t.o01 = (ly.i0 - g.h_lo) * g.fw + (lx.i1 - g.w_lo);
    t.o10 = (ly.i1 - g.h_lo) * g.fw + (lx.i0 - g.w_lo);
    t.o11 = (ly.i1 - g.h_lo) * g.fw + (lx.i1 - g.w_lo);
    t.w00 = ly.l0 * lx.l0; t.w01 = ly.l0 * lx.l1; t.w10 = ly.l1 * lx.l0; t.w11 = ly.l1 * lx.l1;
    return t;
}

template <typename T>
__global__ void __launch_bounds__(kUTW * kUTH) upsample4_soft_argmin_fwd_kernel(
    const T* __restrict__ low, float* __restrict__ disp, float* __restrict__ stats, int Dq, int Hq, int Wq, int H,
    int W, float sh, float sw, int FHW, int64_t total) {
    extern __shared__ float tile[];
    const int b = blockIdx.z;
    const TileGeom tg = tile_geom(sh, sw, Hq, Wq, H, W);
    load_tile(low, tile, b, Dq, Hq, Wq, tg.h_lo, tg.w_lo, tg.fh, tg.fw, FHW);
    __syncthreads();
    const int x = blockIdx.x * kUTW + threadIdx.x, y = blockIdx.y * kUTH + threadIdx.y;
    if (x >= W || y >= H) return;
    const Taps t = make_taps(sh, sw, y, x, Hq, Wq, tg);
    const int D = 4 * Dq;

    float va = bil(tile, t);
    float m = va;                  // d = 0, 1 sample plane 0 exactly
    double s = 2.0, ws = 1.0;      // e = 1 at d = 0 and d = 1
    // interval sums are collected in fp32 and flushed to the fp64 running sums every 8 intervals (and
    // before a rescale): conversions share the MUFU/XU pipe with the 192 ex2 per pixel that bound this kernel
    float fs = 0.f, fw = 0.f;
    const float* pl = tile;
    for (int q = 0; q + 1 < Dq; ++q) {
        pl += FHW;
        const float vb = bil(pl, t);
        const float diff = vb - va;
        const float l0 = fmaf(0.125f, diff, va), l1 = fmaf(0.375f, diff, va);
        const float l2 = fmaf(0.625f, diff, va), l3 = fmaf(0.875f, diff, va);
        const float cm = fmaxf(l0, l3);
        if (cm > m || (q & 7) == 7) {
            s += (double)fs;
            ws += (double)fw;
            fs = 0.f;
            fw = 0.f;
            if (cm > m) {
                const double sc = (double)fast_ex2((m - cm) * kLog2eU);
                s *= sc;
                ws *= sc;
                m = cm;
            }
        }
        const float e0 = fast_ex2((l0 - m) * kLog2eU), e1 = fast_ex2((l1 - m) * kLog2eU);
        const float e2 = fast_ex2((l2 - m) * kLog2eU), e3 = fast_ex2((l3 - m) * kLog2eU);
        const float es = (e0 + e1) + (e2 + e3);
        const float ew = fmaf(3.0f, e3, fmaf(2.0f, e2, e1));
        fs += es;
        fw += fmaf((float)(4 * q + 2), es, ew);
        va = vb;
    }
    s += (double)fs;
    ws += (double)fw;
    {   // d = D-2, D-1 sample plane Dq-1 exactly
        if (va > m) {
            const double sc = (double)fast_ex2((m - va) * kLog2eU);
            s *= sc;
            ws *= sc;
            m = va;
        }
        const double e = (double)fast_ex2((va - m) * kLog2eU);
        s += 2.0 * e;
        ws += e * (double)(2 * D - 3);
    }
    const size_t pix = ((size_t)b * H + y) * W + x;
    disp[pix] = (float)(ws / s);
    if (stats != nullptr) {
        stats[pix] = m;
        stats[total + pix] = log2f((float)s);
    }
}

// ------------------------------------------------------------------------------------------
// Scale exactly 4 along depth AND width (D == 4*Dq, W == 4*Wq: what PSMNet runs, psmnet.py:186-211),
// any vertical upsampling factor.  Round 1's kernel above spent 4 ex2 and ~45 issue slots per pixel and
// depth interval (ncu: issue 80 %, XU 66 %).  This form cuts both:
//   * a thread owns the FOUR output columns x = 4c+2 .. 4c+5 that share the low-res column pair
//     (c, c+1): per plane it reads four taps, blends them vertically once (one packed FFMA2 + FMUL2)
//     and expands to its four pixels with the constant weights {1/8, 3/8, 5/8, 7/8} (two FFMA2);
//   * within a depth interval the four logits are an arithmetic progression x0 + k*diff/4, so the
//     four exponentials are a geometric one: e_start = 2^((max(l0,l3) - m)*log2e) at the end nearer
//     the running max and ratio r = 2^(-|diff|/4*log2e) <= 1 -- two ex2 and three multiplies;
//   * everything per pixel pair is packed fp32x2 (FFMA2 / FADD2 / FMUL2).
//   * two passes over the shared-memory tile: first the exact per-pixel maximum (max over the Dq
//     interpolated planes), then the sums against that fixed reference -- no rescale and no data-dependent
//     branch in the hot loop;
// Interval sums are collected in fp32 relative to the first depth of the current block of 8 intervals and
// flushed to the fp64 running sums at the end of the block.
// ------------------------------------------------------------------------------------------
typedef unsigned long long u64u;
__device__ __forceinline__ u64u upk2f(float lo, float hi) { u64u r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void uunpk(u64u v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ u64u uadd(u64u a, u64u b) { u64u r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ u64u usub(u64u a, u64u b) { u64u r; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ u64u umul(u64u a, u64u b) { u64u r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ u64u ufma(u64u a, u64u b, u64u c) { u64u r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }

constexpr int kU4G = 32, kU4H = 8;  // groups (of 4 output columns) x rows per CTA
constexpr int kU4FW = kU4G + 1;     // low-res columns under a tile (taps c and c+1)

// values of the thread's four pixels on low-res plane `pl`: (v0,v1) and (v2,v3)
__device__ __forceinline__ void bil4(const float* __restrict__ pl, int oa, int ob, u64u ly0, u64u ly1, u64u& v01,
                                     u64u& v23) {
    const u64u top = upk2f(pl[oa], pl[oa + 1]), bot = upk2f(pl[ob], pl[ob + 1]);
    const u64u col = ufma(bot, ly1, umul(top, ly0));  // (colA, colB): vertical blend of the two tap columns
    float ca, cb;
    uunpk(col, ca, cb);
    const float dc = cb - ca;
    const u64u dc2 = upk2f(dc, dc), ca2 = upk2f(ca, ca);
    v01 = ufma(upk2f(0.125f, 0.375f), dc2, ca2);
    v23 = ufma(upk2f(0.625f, 0.875f), dc2, ca2);
}

// grid = (ceil((Wq + 1) / 32), ceil(H / 8), B), block = (32, 8).  smem: tile[Dq][fh][33]
template <typename T>
__global__ void __launch_bounds__(kU4G * kU4H) upsample4x_soft_argmin_fwd_kernel(
    const T* __restrict__ low, float* __restrict__ disp, float* __restrict__ stats, int Dq, int Hq, int Wq, int H,
    float sh, int fh_cap, int64_t total) {
    extern __shared__ float tile[];
    const int b = blockIdx.z, W = 4 * Wq;
    const int c0 = blockIdx.x * kU4G - 1;  // first group of the tile (group -1 holds x = 0, 1)
    const int y0 = blockIdx.y * kU4H, y1 = min(y0 + kU4H, H) - 1;
    const int h_lo = src_index(sh, y0, Hq).i0, h_hi = src_index(sh, y1, Hq).i1;
    const int fh = h_hi - h_lo + 1;
    const int FHW = fh_cap * kU4FW;
    {   // footprint, column / row indices clamped so that edge groups read a repeated column (=> weightless lerp)
        const int tid = threadIdx.y * kU4G + threadIdx.x;
        const int npos = fh * kU4FW;
        const size_t plane = (size_t)Hq * Wq;
        for (int pos = tid & 63; pos < npos; pos += 64) {
            const int hh = pos / kU4FW, ww = pos - hh * kU4FW;
            const int col = min(max(c0 + ww, 0), Wq - 1);
            const T* srcp = low + (size_t)b * Dq * plane + (size_t)(h_lo + hh) * Wq + col;
            for (int q = tid >> 6; q < Dq; q += (kU4G * kU4H) >> 6) tile[q * FHW + pos] = ld_f32(srcp + (size_t)q * plane);
        }
    }
    __syncthreads();
    const int y = y0 + threadIdx.y;
    const int c = c0 + threadIdx.x;
    const int xbase = 4 * c + 2;
    if (y >= H || xbase >= W) return;
    const Lerp ly = src_index(sh, y, Hq);
    const int oa = (ly.i0 - h_lo) * kU4FW + threadIdx.x, ob = (ly.i1 - h_lo) * kU4FW + threadIdx.x;
    const u64u ly0 = upk2f(ly.l0, ly.l0), ly1 = upk2f(ly.l1, ly.l1);
    const int D = 4 * Dq;
    const float kQ = -0.25f * kLog2eU;

    // pass 1: the exact maximum of every pixel's D logits.  The samples of interval q lie at 1/8 .. 7/8 between
    // planes q and q+1 (a lerp is monotone: the interval's maximum is its first or last sample), d = 0, 1 sample
    // plane 0 and d = D-2, D-1 plane Dq-1 exactly.  (The maximum over the PLANES would not do: with logits in the
    // thousands every sample can sit hundreds below the nearest plane and all exponentials would underflow.)
    // With the reference fixed up front, pass 2 has no rescale, no data-dependent branch (round 1's one-pass form
    // took its fp64 flush-and-rescale branch on almost every interval of almost every warp) and no per-interval
    // float->double conversion.
    float m[4];
    {
        u64u pa[2], pb[2];
        bil4(tile, oa, ob, ly0, ly1, pa[0], pa[1]);
        uunpk(pa[0], m[0], m[1]);
        uunpk(pa[1], m[2], m[3]);
        const float* pq = tile;
        for (int q = 1; q < Dq; ++q) {
            pq += FHW;
            bil4(pq, oa, ob, ly0, ly1, pb[0], pb[1]);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const u64u diff = usub(pb[h], pa[h]);
                float a0, a1, b0, b1;
                uunpk(ufma(upk2f(0.125f, 0.125f), diff, pa[h]), a0, a1);
                uunpk(ufma(upk2f(0.875f, 0.875f), diff, pa[h]), b0, b1);
                m[2 * h] = fmaxf(m[2 * h], fmaxf(a0, b0));
                m[2 * h + 1] = fmaxf(m[2 * h + 1], fmaxf(a1, b1));
                pa[h] = pb[h];
            }
        }
        float l0, l1, l2, l3;
        uunpk(pa[0], l0, l1);
        uunpk(pa[1], l2, l3);
        m[0] = fmaxf(m[0], l0);
        m[1] = fmaxf(m[1], l1);
        m[2] = fmaxf(m[2], l2);
        m[3] = fmaxf(m[3], l3);
    }
    const u64u m2[2] = {upk2f(m[0], m[1]), upk2f(m[2], m[3])};
    const u64u kL2 = upk2f(kLog2eU, kLog2eU);

    // pass 2
    u64u va[2];
    bil4(tile, oa, ob, ly0, ly1, va[0], va[1]);
    double s[4], ws[4];
    {   // d = 0, 1 sample plane 0 exactly
        float e[4], t0, t1;
        uunpk(umul(usub(va[0], m2[0]), kL2), t0, t1);
        e[0] = fast_ex2(t0);
        e[1] = fast_ex2(t1);
        uunpk(umul(usub(va[1], m2[1]), kL2), t0, t1);
        e[2] = fast_ex2(t0);
        e[3] = fast_ex2(t1);
#pragma unroll
        for (int j = 0; j < 4; ++j) { s[j] = 2.0 * (double)e[j]; ws[j] = (double)e[j]; }
    }
    u64u fs[2] = {0ull, 0ull}, fw[2] = {0ull, 0ull};  // block sums: sum e, sum (d - dblk) e over <= 8 intervals
    int qb = 0;                                      // first interval of the current block
    const float* pl = tile;
    for (int q = 0; q + 1 < Dq; ++q) {
        pl += FHW;
        u64u vb[2];
        bil4(pl, oa, ob, ly0, ly1, vb[0], vb[1]);
        const float ofs = (float)(4 * (q - qb));
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const u64u diff = usub(vb[h], va[h]);
            const u64u l0 = ufma(upk2f(0.125f, 0.125f), diff, va[h]), l3 = ufma(upk2f(0.875f, 0.875f), diff, va[h]);
            float l0a, l0b, l3a, l3b, da, db, ta, tb;
            uunpk(l0, l0a, l0b);
            uunpk(l3, l3a, l3b);
            uunpk(diff, da, db);
            // geometric progression from the end nearer the max: e_start, then ratio r = 2^(-|diff|/4 log2e) <= 1
            uunpk(umul(usub(upk2f(fmaxf(l0a, l3a), fmaxf(l0b, l3b)), m2[h]), kL2), ta, tb);
            const u64u es = upk2f(fast_ex2(ta), fast_ex2(tb));
            const u64u r = upk2f(fast_ex2(fabsf(da) * kQ), fast_ex2(fabsf(db) * kQ));
            const u64u f1 = umul(es, r), f2 = umul(f1, r), f3 = umul(f2, r);
            const u64u sum = uadd(uadd(es, f1), uadd(f2, f3));
            // sum_k k e_k: es is e_3 when diff >= 0 (3 es + 2 f1 + f2), e_0 otherwise (f1 + 2 f2 + 3 f3)
            const u64u wup = ufma(upk2f(3.f, 3.f), es, ufma(upk2f(2.f, 2.f), f1, f2));
            const u64u wdn = ufma(upk2f(3.f, 3.f), f3, ufma(upk2f(2.f, 2.f), f2, f1));
            float wua, wub, wda, wdb;
            uunpk(wup, wua, wub);
            uunpk(wdn, wda, wdb);
            const u64u ew = upk2f(da >= 0.f ? wua : wda, db >= 0.f ? wub : wdb);
            fs[h] = uadd(fs[h], sum);
            fw[h] = uadd(fw[h], ufma(upk2f(ofs, ofs), sum, ew));
            va[h] = vb[h];
        }
        if (q - qb == 7 || q + 2 == Dq) {  // uniform: flush the block into the fp64 running sums
            const double base = (double)(4 * qb + 2);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                float fsa, fsb, fwa, fwb;
                uunpk(fs[h], fsa, fsb);
                uunpk(fw[h], fwa, fwb);
                s[2 * h] += (double)fsa;
                s[2 * h + 1] += (double)fsb;
                ws[2 * h] += fma(base, (double)fsa, (double)fwa);
                ws[2 * h + 1] += fma(base, (double)fsb, (double)fwb);
                fs[h] = 0ull;
                fw[h] = 0ull;
            }
            qb = q + 1;
        }
    }
    float o[4], l2[4];
    {   // d = D-2, D-1 sample plane Dq-1 exactly
        float vl[4], t0, t1;
        uunpk(umul(usub(va[0], m2[0]), kL2), t0, t1);
        vl[0] = fast_ex2(t0);
        vl[1] = fast_ex2(t1);
        uunpk(umul(usub(va[1], m2[1]), kL2), t0, t1);
        vl[2] = fast_ex2(t0);
        vl[3] = fast_ex2(t1);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const double e = (double)vl[j];
            s[j] += 2.0 * e;
            ws[j] += e * (double)(2 * D - 3);
            o[j] = (float)(ws[j] / s[j]);
            l2[j] = log2f((float)s[j]);
        }
    }
    const size_t row = ((size_t)b * H + y) * W;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int x = xbase + 2 * h;
        if (x < 0 || x >= W) continue;  // W = 4*Wq and x is even: a pair is wholly inside or outside
        *reinterpret_cast<float2*>(disp + row + x) = make_float2(o[2 * h], o[2 * h + 1]);
        if (stats != nullptr) {
            *reinterpret_cast<float2*>(stats + row + x) = make_float2(m[2 * h], m[2 * h + 1]);
            *reinterpret_cast<float2*>(stats + total + row + x) = make_float2(l2[2 * h], l2[2 * h + 1]);
        }
    }
}

template <typename T>
__global__ void __launch_bounds__(kUTW * kUTH) upsample4_soft_argmin_bwd_pix_kernel(
    const T* __restrict__ low, const float* __restrict__ disp, const float* __restrict__ stats,
    const float* __restrict__ gdisp, float* __restrict__ G, int Dq, int Hq, int Wq, int H, int W, float sh, float sw,
    int FHW, int64_t total) {
    extern __shared__ float tile[];
    const int b = blockIdx.z;
    const TileGeom tg = tile_geom(sh, sw, Hq, Wq, H, W);
    load_tile(low, tile, b, Dq, Hq, Wq, tg.h_lo, tg.w_lo, tg.fh, tg.fw, FHW);
    __syncthreads();
    const int x = blockIdx.x * kUTW + threadIdx.x, y = blockIdx.y * kUTH + threadIdx.y;
    if (x >= W || y >= H) return;
    const Taps t = make_taps(sh, sw, y, x, Hq, Wq, tg);
    const int D = 4 * Dq;
    const size_t pix = ((size_t)b * H + y) * W + x;
    const float m = stats[pix], l2s = stats[total + pix], out = disp[pix], g = gdisp[pix];
    const size_t HW = (size_t)H * W;
    float* Gp = G + (size_t)b * Dq * HW + (size_t)y * W + x;

    float va = bil(tile, t);
    // d = 0, 1 -> plane 0 with weight 1
    float carry;
    {
        const float p = fast_ex2(fmaf(va - m, kLog2eU, -l2s));
        carry = p * g * ((0.0f - out) + (1.0f - out));
    }
    const float* pl = tile;
    for (int q = 0; q + 1 < Dq; ++q) {
        pl += FHW;
        const float vb = bil(pl, t);
        const float diff = vb - va;
        const float bo = (float)(4 * q + 2) - out;
        const float p0 = fast_ex2(fmaf(fmaf(0.125f, diff, va) - m, kLog2eU, -l2s));
        const float p1 = fast_ex2(fmaf(fmaf(0.375f, diff, va) - m, kLog2eU, -l2s));
        const float p2 = fast_ex2(fmaf(fmaf(0.625f, diff, va) - m, kLog2eU, -l2s));
        const float p3 = fast_ex2(fmaf(fmaf(0.875f, diff, va) - m, kLog2eU, -l2s));
        const float g0 = p0 * (bo * g), g1 = p1 * ((bo + 1.0f) * g);
        const float g2 = p2 * ((bo + 2.0f) * g), g3 = p3 * ((bo + 3.0f) * g);
        const float gb = fmaf(0.875f, g3, fmaf(0.625f, g2, fmaf(0.375f, g1, 0.125f * g0)));
        const float gs = (g0 + g1) + (g2 + g3);
        Gp[(size_t)q * HW] = carry + (gs - gb);
        carry = gb;
        va = vb;
    }
    {   // d = D-2, D-1 -> plane Dq-1 with weight 1
        const float p = fast_ex2(fmaf(va - m, kLog2eU, -l2s));
        Gp[(size_t)(Dq - 1) * HW] = carry + p * g * (((float)(D - 2) - out) + ((float)(D - 1) - out));
    }
}

// backward stage 2: T[b,q,y,w] = sum_x wx(x,w) * G[b,q,y,x].
// The tap weights of a low-res column depend on w only: each thread computes its <= kMaxTaps weights once
// and applies them to kRowsPerCta rows.  grid = (ceil(Wq/128), ceil(H/kRowsPerCta), B*Dq)
constexpr int kMaxTaps = 16, kRowsPerCta = 8;

__device__ __forceinline__ void tap_range(float scale, int w, int out_size, int& lo, int& hi) {
    const float inv = 1.0f / scale;  // output indices whose source index can touch w: src in (w-1, w+1)
    lo = max((int)floorf(((float)w - 1.0f + 0.5f) * inv - 0.5f) - 1, 0);
    hi = min((int)ceilf(((float)w + 1.0f + 0.5f) * inv - 0.5f) + 1, out_size - 1);
}

__device__ __forceinline__ float tap_weight(float scale, int x, int w, int in_size) {
    const Lerp l = src_index(scale, x, in_size);
    float wt = 0.f;
    if (l.i0 == w) wt += l.l0;
    if (l.i1 == w) wt += l.l1;
    return wt;
}

__global__ void __launch_bounds__(128) upsample_bwd_reduce_x_kernel(const float* __restrict__ G, float* __restrict__ T,
                                                                   int H, int W, int Wq, float sw) {
    const int w = blockIdx.x * 128 + threadIdx.x;
    if (w >= Wq) return;
    int xlo, xhi;
    tap_range(sw, w, W, xlo, xhi);
    // drop zero-weight taps at both ends so that the window fits kMaxTaps (the host checks the bound)
    while (xlo < xhi && tap_weight(sw, xlo, w, Wq) == 0.f) ++xlo;
    while (xhi > xlo && tap_weight(sw, xhi, w, Wq) == 0.f) --xhi;
    float wt[kMaxTaps];
#pragma unroll
    for (int t = 0; t < kMaxTaps; ++t) wt[t] = (xlo + t <= xhi) ? tap_weight(sw, xlo + t, w, Wq) : 0.f;
    const int y0 = blockIdx.y * kRowsPerCta;
    const int y1 = min(y0 + kRowsPerCta, H);
    for (int y = y0; y < y1; ++y) {
        const size_t row = (size_t)blockIdx.z * H + y;
        const float* g = G + row * W + xlo;
        float acc = 0.f;
#pragma unroll
        for (int t = 0; t < kMaxTaps; ++t)
            if (xlo + t <= xhi) acc = fmaf(wt[t], __ldg(g + t), acc);
        T[row * Wq + w] = acc;
    }
}

// backward stage 3: glow[b,q,h,w] = sum_y wy(y,h) * T[b,q,y,w].   grid = (ceil(Wq/128), Hq, B*Dq)
// glow of 16 bits: the fp32 sum is rounded once, to nearest even, at the store.
template <typename O>
__global__ void __launch_bounds__(128) upsample_bwd_reduce_y_kernel(const float* __restrict__ T, O* __restrict__ glow,
                                                                   int H, int Hq, int Wq, float sh) {
    const int w = blockIdx.x * 128 + threadIdx.x;
    if (w >= Wq) return;
    const int h = blockIdx.y;
    const size_t plane = blockIdx.z;
    const float inv = 1.0f / sh;
    int ylo = (int)floorf(((float)h - 1.0f + 0.5f) * inv - 0.5f) - 1;
    int yhi = (int)ceilf(((float)h + 1.0f + 0.5f) * inv - 0.5f) + 1;
    ylo = max(ylo, 0);
    yhi = min(yhi, H - 1);
    float acc = 0.f;
    for (int y = ylo; y <= yhi; ++y) {
        const Lerp l = src_index(sh, y, Hq);
        float wt = 0.f;
        if (l.i0 == h) wt += l.l0;
        if (l.i1 == h) wt += l.l1;
        if (wt != 0.f) acc = fmaf(wt, __ldg(T + (plane * H + y) * Wq + w), acc);
    }
    st_from_f32(glow + (plane * Hq + h) * Wq + w, acc);
}

static int tile_extent(int in_size, int out_size, int tile) {
    // max number of low-res indices under `tile` consecutive outputs (+1 for the i1 neighbour)
    const double scale = (double)in_size / out_size;
    int e = (int)(tile * scale) + 3;
    return e < in_size ? e : in_size;
}

}  // namespace az

using namespace az;

extern "C" int64_t az_upsample_soft_argmin_workspace_bytes(int64_t B, int64_t Dq, int64_t H, int64_t W, int64_t Wq) {
    return B * Dq * H * (W + Wq) * (int64_t)sizeof(float);
}

static int upsample_args_ok(int64_t B, int64_t Dq, int64_t Hq, int64_t Wq, int64_t D, int64_t H, int64_t W) {
    if (B <= 0 || Dq <= 0 || Hq <= 0 || Wq <= 0 || D <= 0 || H <= 0 || W <= 0) return 0;
    if (D < Dq || H < Hq || W < Wq) return 0;  // upsampling only
    if (B > 65535 || H > 65535 || B * Dq > 65535 || H * W >= (1ll << 31)) return 0;
    if (2.0 * (double)W / (double)Wq + 3.0 > kMaxTaps) return 0;  // horizontal factor <= 6: the backward's tap window
    return 1;
}

// fp32 (knob = the AZ_USA_FWD developer knob) and 16-bit low-res logits (knob = 1, the default: the kernel choice is a
// function of the shape alone, as for fp32 at the default).
template <typename T>
static int upsample_fwd(const T* lowres, float* disp, float* stats, int64_t B, int64_t Dq, int64_t Hq, int64_t Wq,
                        int64_t D, int64_t H, int64_t W, int knob, cudaStream_t stream) {
    const int fh = tile_extent((int)Hq, (int)H, kUTH), fw = tile_extent((int)Wq, (int)W, kUTW);
    const int FHW = fh * fw;
    const size_t smem = ((size_t)Dq * FHW + D + Dq + 1) * sizeof(float);
    if (smem > 200 * 1024) return AZ_ERR_BAD_ARG;
    cudaError_t e = cudaFuncSetAttribute(upsample_soft_argmin_fwd_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         200 * 1024);
    if (e != cudaSuccess) return (int)e;
    dim3 grid((unsigned)ceil_div(W, kUTW), (unsigned)ceil_div(H, kUTH), (unsigned)B);
    if (D == 4 * Dq && Dq >= 2 && W == 4 * Wq && knob == 1) {
        // x4 in depth and width (PSMNet): 4 pixels per thread, packed arithmetic, 2 ex2 per interval
        const int fh4 = tile_extent((int)Hq, (int)H, kU4H);
        const size_t smem4 = (size_t)Dq * fh4 * kU4FW * sizeof(float);
        if (smem4 <= 200 * 1024) {
            e = cudaFuncSetAttribute(upsample4x_soft_argmin_fwd_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     200 * 1024);
            if (e != cudaSuccess) return (int)e;
            dim3 g4((unsigned)ceil_div(Wq + 1, kU4G), (unsigned)ceil_div(H, kU4H), (unsigned)B);
            upsample4x_soft_argmin_fwd_kernel<T><<<g4, dim3(kU4G, kU4H), smem4, stream>>>(
                lowres, disp, stats, (int)Dq, (int)Hq, (int)Wq, (int)H, (float)Hq / (float)H, fh4, B * H * W);
            AZ_LAUNCH_CHECK();
            return 0;
        }
    }
    if (D == 4 * Dq && Dq >= 2) {
        e = cudaFuncSetAttribute(upsample4_soft_argmin_fwd_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 200 * 1024);
        if (e != cudaSuccess) return (int)e;
        upsample4_soft_argmin_fwd_kernel<T><<<grid, dim3(kUTW, kUTH), smem, stream>>>(
            lowres, disp, stats, (int)Dq, (int)Hq, (int)Wq, (int)H, (int)W, (float)Hq / (float)H, (float)Wq / (float)W,
            FHW, B * H * W);
        AZ_LAUNCH_CHECK();
        return 0;
    }
    upsample_soft_argmin_fwd_kernel<T><<<grid, dim3(kUTW, kUTH), smem, stream>>>(
        lowres, disp, stats, (int)Dq, (int)Hq, (int)Wq, (int)D, (int)H, (int)W, (float)Dq / (float)D,
        (float)Hq / (float)H, (float)Wq / (float)W, FHW, B * H * W);
    AZ_LAUNCH_CHECK();
    return 0;
}

template <typename T>
static int upsample_bwd(const T* lowres, const float* disp, const float* stats, const float* gdisp, T* glow,
                        void* workspace, int64_t B, int64_t Dq, int64_t Hq, int64_t Wq, int64_t D, int64_t H, int64_t W,
                        cudaStream_t st) {
    const int fh = tile_extent((int)Hq, (int)H, kUTH), fw = tile_extent((int)Wq, (int)W, kUTW);
    const int FHW = fh * fw;
    const size_t smem = ((size_t)Dq * FHW + D + Dq + 1) * sizeof(float);
    if (smem > 200 * 1024) return AZ_ERR_BAD_ARG;
    cudaError_t e = cudaFuncSetAttribute(upsample_soft_argmin_bwd_pix_kernel<T>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    if (e != cudaSuccess) return (int)e;
    float* G = (float*)workspace;
    float* Tw = G + B * Dq * H * W;
    const float sd = (float)Dq / (float)D, sh = (float)Hq / (float)H, sw = (float)Wq / (float)W;
    dim3 grid((unsigned)ceil_div(W, kUTW), (unsigned)ceil_div(H, kUTH), (unsigned)B);
    if (D == 4 * Dq && Dq >= 2) {
        e = cudaFuncSetAttribute(upsample4_soft_argmin_bwd_pix_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 200 * 1024);
        if (e != cudaSuccess) return (int)e;
        upsample4_soft_argmin_bwd_pix_kernel<T><<<grid, dim3(kUTW, kUTH), smem, st>>>(
            lowres, disp, stats, gdisp, G, (int)Dq, (int)Hq, (int)Wq, (int)H, (int)W, sh, sw, FHW, B * H * W);
    } else {
        upsample_soft_argmin_bwd_pix_kernel<T><<<grid, dim3(kUTW, kUTH), smem, st>>>(
            lowres, disp, stats, gdisp, G, (int)Dq, (int)Hq, (int)Wq, (int)D, (int)H, (int)W, sd, sh, sw, FHW,
            B * H * W);
    }
    AZ_LAUNCH_CHECK();
    dim3 gx((unsigned)ceil_div(Wq, 128), (unsigned)ceil_div(H, kRowsPerCta), (unsigned)(B * Dq));
    upsample_bwd_reduce_x_kernel<<<gx, 128, 0, st>>>(G, Tw, (int)H, (int)W, (int)Wq, sw);
    AZ_LAUNCH_CHECK();
    dim3 gy((unsigned)ceil_div(Wq, 128), (unsigned)Hq, (unsigned)(B * Dq));
    upsample_bwd_reduce_y_kernel<T><<<gy, 128, 0, st>>>(Tw, glow, (int)H, (int)Hq, (int)Wq, sh);
    AZ_LAUNCH_CHECK();
    return 0;
}

extern "C" int az_upsample_soft_argmin_fwd(const float* lowres, float* disp, float* stats, int64_t B, int64_t Dq,
                                           int64_t Hq, int64_t Wq, int64_t D, int64_t H, int64_t W, void* stream) {
    if (!lowres || !disp || !upsample_args_ok(B, Dq, Hq, Wq, D, H, W)) return AZ_ERR_BAD_ARG;
    return upsample_fwd(lowres, disp, stats, B, Dq, Hq, Wq, D, H, W, az::tuning("AZ_USA_FWD", 1), (cudaStream_t)stream);
}

extern "C" int az_upsample_soft_argmin_bwd(const float* lowres, const float* disp, const float* stats,
                                           const float* gdisp, float* glow, void* workspace, int64_t B, int64_t Dq,
                                           int64_t Hq, int64_t Wq, int64_t D, int64_t H, int64_t W, void* stream) {
    if (!lowres || !disp || !stats || !gdisp || !glow || !workspace || !upsample_args_ok(B, Dq, Hq, Wq, D, H, W))
        return AZ_ERR_BAD_ARG;
    return upsample_bwd(lowres, disp, stats, gdisp, glow, workspace, B, Dq, Hq, Wq, D, H, W, (cudaStream_t)stream);
}

extern "C" int az_upsample_soft_argmin_fwd_16(const void* lowres, float* disp, float* stats, int64_t B, int64_t Dq,
                                              int64_t Hq, int64_t Wq, int64_t D, int64_t H, int64_t W, int dtype,
                                              void* stream) {
    if (!lowres || !disp || !upsample_args_ok(B, Dq, Hq, Wq, D, H, W)) return AZ_ERR_BAD_ARG;
    if (dtype == AZ_DTYPE_BF16)
        return upsample_fwd(static_cast<const __nv_bfloat16*>(lowres), disp, stats, B, Dq, Hq, Wq, D, H, W, 1,
                            (cudaStream_t)stream);
    if (dtype == AZ_DTYPE_F16)
        return upsample_fwd(static_cast<const __half*>(lowres), disp, stats, B, Dq, Hq, Wq, D, H, W, 1,
                            (cudaStream_t)stream);
    return AZ_ERR_BAD_ARG;
}

extern "C" int az_upsample_soft_argmin_bwd_16(const void* lowres, const float* disp, const float* stats,
                                              const float* gdisp, void* glow, void* workspace, int64_t B, int64_t Dq,
                                              int64_t Hq, int64_t Wq, int64_t D, int64_t H, int64_t W, int dtype,
                                              void* stream) {
    if (!lowres || !disp || !stats || !gdisp || !glow || !workspace || !upsample_args_ok(B, Dq, Hq, Wq, D, H, W))
        return AZ_ERR_BAD_ARG;
    if (dtype == AZ_DTYPE_BF16)
        return upsample_bwd(static_cast<const __nv_bfloat16*>(lowres), disp, stats, gdisp,
                            static_cast<__nv_bfloat16*>(glow), workspace, B, Dq, Hq, Wq, D, H, W, (cudaStream_t)stream);
    if (dtype == AZ_DTYPE_F16)
        return upsample_bwd(static_cast<const __half*>(lowres), disp, stats, gdisp, static_cast<__half*>(glow),
                            workspace, B, Dq, Hq, Wq, D, H, W, (cudaStream_t)stream);
    return AZ_ERR_BAD_ARG;
}
