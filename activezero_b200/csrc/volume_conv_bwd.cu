// Backward of the first aggregation convolution on the IMPLICIT concat volume (the forward is volume_conv_v2.cu):
//   out = conv3d(V, W, padding 1),  V[c,i,y,x] = L[c,y,x]·[x>=i],  V[32+c,i,y,x] = R[c,y,x-i]·[x>=i]
// with g = dLoss/d out [B,32,Dq,H,W].  The convolution is linear and the features have no disparity axis, so every
// gradient reduces g over d first and only then contracts with the weights; the volume's gradient never exists.
// For the nine (kd, kx) taps, lo = max(0, 1-kd), hi = min(Dq-1, Dq-kd):
//   A[kd,kx][o,y,x] = sum_{d=lo}^{min(x+kx-kd, hi)} g[o,d,y,x]                       (prefix sum down a column)
//   Z[kd,kx][o,y,u] = sum_{d=lo}^{hi} g[o,d,y,u+d+kd-kx],  0 <= u+d+kd-kx <= min(W-1, W-kx)   (sum along a diagonal)
//   dL[c,y',x'] = sum_{o,kd,ky,kx} W[o,c,kd,ky,kx]    · A[kd,kx][o,y'-ky+1,x'-kx+1]   (zero outside the image)
//   dR[c,y',u]  = sum_{o,kd,ky,kx} W[o,32+c,kd,ky,kx] · Z[kd,kx][o,y'-ky+1,u]
//   dW[o,c,kd,ky,kx]    = sum_{b,y',x'} A[kd,kx][b,o,y'-ky+1,x'-kx+1] · L[b,c,y',x']
//   dW[o,32+c,kd,ky,kx] = sum_{b,y',u}  Z[kd,kx][b,o,y'-ky+1,u]       · R[b,c,y',u]
// The contractions are 1/Dq of the FLOPs of dgrad + wgrad on the materialised volume, so they stay in fp32 on the
// CUDA cores.  Four kernels, all gather-style with fixed summation orders and no atomics (bit-identical run to run):
//   1. reduce  : streams g once and writes the 18 planes A[kd,kx], Z[kd,kx] ([B,32,H,W] each) to the workspace
//   2. dfeat   : dL / dR, a 27-tap 32 -> 32-channel contraction of the shifted planes (8 x 4 register tile per thread)
//   3. wgrad   : per-CTA partial sums of the 54 outer products over a chunk of image rows, into the workspace
//   4. finalize: dW = the partials added in chunk order
// The kernels are templated on the element types of g, the features and their gradients (float, bf16, fp16) and of
// the weight and dW (float or the features' 16-bit type).  A 16-bit value is widened exactly where it is read, the
// planes, the partials and every accumulator stay fp32 in the same order, and a 16-bit result is rounded once, to
// nearest even, at its store: the 16-bit backward equals the fp32 one on the widened inputs followed by .to(dtype).
#include <type_traits>

#include "common.cuh"

namespace az {

constexpr int kVbC = 32;           // feature channels per half (PSMNet)
constexpr int kVbPlanes = 18;      // A[kd,kx] (0..8), Z[kd,kx] (9..17)
constexpr int kVbRedT = 128;       // reduce: threads per CTA (one column each; two in vcb_reduce2_kernel)
constexpr int kVbTX = 128;         // dfeat: output columns per CTA (128 threads, 4 columns x 8 channels each)
constexpr int kVbDfSmem = (3 * kVbC * kVbTX + 3 * kVbC * kVbC) * 4;   // 61 440
constexpr int kVwT = 192, kVwTX = 32, kVwP = 36;   // wgrad: threads, positions per tile, smem pitch of a position
constexpr int kVwChunks = 64;      // target number of row chunks (CTAs per plane) of the weight gradient

__host__ __device__ inline int64_t vcb_rows_per_chunk(int64_t B, int64_t H) { return ceil_div(B * H, kVwChunks); }
__host__ __device__ inline int64_t vcb_nchunks(int64_t B, int64_t H) { return ceil_div(B * H, vcb_rows_per_chunk(B, H)); }

// ------------------------------------------------------------------------------------------
// 1. reduce.  grid = (B*32*H rows, ceil(W / kVbRedT)), kVbRedT threads; thread j owns column x = u = u0 + j.
// A: with M(e) = sum_{d=1}^{e} g[d] (planes 1 .. Dq-2 only), g0 = g[0], gl = g[Dq-1] (0 when Dq = 1) and s = kx - kd,
//   kd = 0: M(min(x+s, Dq-2)) + gl·[x+s >= Dq-1]
//   kd = 1: [x+s >= 0] · ((g0 + M(min(x+s, Dq-2))) + gl·[x+s >= Dq-1])
//   kd = 2: [x+s >= 0, Dq >= 2] · (g0 + M(min(x+s, Dq-2)))
//   one pass down the column: plain accumulation up to plane x-3, then the five snapshots s = -2..2 unrolled.
// Z: with the core diagonal Dg(v) = sum_{d=max(1,-v)}^{min(Dq-2, W-2-v)} g[d][v+d] (shared by all taps), t = kd - kx,
//   v = u + t and xmax = W - 1 - [kx == 2]:
//   Z = ((Dg(v) + g[0][v]·[kd = 1 or (kd = 2, Dq >= 2), 0 <= v <= xmax])
//             + g[Dq-1][v+Dq-1]·[kd <= 1, Dq >= 2, 0 <= v+Dq-1 <= xmax])
//             + g[W-1-v][W-1]·[kx <= 1, 1 <= W-1-v <= Dq-2]
//   the CTA computes Dg for v = u0-2 .. u0+kVbRedT+1 into shared memory first.
// ------------------------------------------------------------------------------------------
template <typename TG>
__global__ void __launch_bounds__(kVbRedT) vcb_reduce_kernel(const TG* __restrict__ g, float* __restrict__ planes,
                                                             int B, int H, int W, int Dq) {
    __shared__ float dg[kVbRedT + 4];
    const int64_t row = blockIdx.x;  // (b*32 + o)*H + y
    const int y = (int)(row % H);
    const int64_t bo = row / H;
    const int u0 = (int)blockIdx.y * kVbRedT;
    const size_t HW = (size_t)H * W;
    const TG* gr = g + (size_t)bo * Dq * HW + (size_t)y * W;  // g[b,o,0,y,0]
    for (int i = threadIdx.x; i < kVbRedT + 4; i += kVbRedT) {
        const int v = u0 - 2 + i;
        const int dlo = max(1, -v), dhi = min(Dq - 2, W - 2 - v);
        float acc = 0.f;
#pragma unroll 8
        for (int d = dlo; d <= dhi; ++d) acc += ld_f32(gr + (size_t)d * HW + (v + d));
        dg[i] = acc;
    }
    __syncthreads();
    const int x = u0 + (int)threadIdx.x;
    if (x >= W) return;
    const TG* gc = gr + x;
    const float g0 = ld_f32(gc);
    const float gl = Dq >= 2 ? ld_f32(gc + (size_t)(Dq - 1) * HW) : 0.f;
    float M = 0.f, snap[5];
    const int e0 = min(x - 3, Dq - 2);
#pragma unroll 8
    for (int d = 1; d <= e0; ++d) M += ld_f32(gc + (size_t)d * HW);
#pragma unroll
    for (int k = 0; k < 5; ++k) {
        const int e = x + k - 2;
        if (e >= 1 && e <= Dq - 2) M += ld_f32(gc + (size_t)e * HW);
        snap[k] = M;
    }
    const size_t NP = (size_t)B * kVbC * HW;  // floats per plane
    float* out = planes + (size_t)row * W + x;
#pragma unroll
    for (int kd = 0; kd < 3; ++kd) {
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
            const int s = kx - kd;
            const float m = snap[s + 2];
            const float last = (x + s >= Dq - 1) ? gl : 0.f;
            float a;
            if (kd == 0) a = m + last;
            else if (kd == 1) a = (x + s >= 0) ? (g0 + m) + last : 0.f;
            else a = (x + s >= 0 && Dq >= 2) ? g0 + m : 0.f;
            out[(size_t)(kd * 3 + kx) * NP] = a;
        }
    }
#pragma unroll
    for (int kd = 0; kd < 3; ++kd) {
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
            const int t = kd - kx, v = x + t, xmax = W - 1 - (kx == 2 ? 1 : 0);
            float z = dg[threadIdx.x + 2 + t];
            if ((kd == 1 || (kd == 2 && Dq >= 2)) && v >= 0 && v <= xmax) z += ld_f32(gr + v);
            const int vl = v + Dq - 1;
            if (kd <= 1 && Dq >= 2 && vl >= 0 && vl <= xmax) z += ld_f32(gr + (size_t)(Dq - 1) * HW + vl);
            const int dw = W - 1 - v;
            if (kx <= 1 && dw >= 1 && dw <= Dq - 2) z += ld_f32(gr + (size_t)dw * HW + (W - 1));
            out[(size_t)(9 + kd * 3 + kx) * NP] = z;
        }
    }
}

// two adjacent 16-bit elements in one 4-byte load (p 4-byte aligned), widened exactly
__device__ __forceinline__ float2 ld2_f32(const __nv_bfloat16* p) {
    return __bfloat1622float2(__ldg(reinterpret_cast<const __nv_bfloat162*>(p)));
}
__device__ __forceinline__ float2 ld2_f32(const __half* p) { return __half22float2(__ldg(reinterpret_cast<const __half2*>(p))); }

// 1b. reduce for 16-bit g with an even W and a 4-byte aligned g: thread j owns the two columns x = u0 + 2j, x + 1 and
// reads both with one 4-byte load per plane, so a warp reads 128 B per plane as the fp32 kernel does.  Each column's
// sums are vcb_reduce_kernel's, term for term and in the same order; the CTA covers 2 * kVbRedT columns.
template <typename TG>
__global__ void __launch_bounds__(kVbRedT) vcb_reduce2_kernel(const TG* __restrict__ g, float* __restrict__ planes,
                                                              int B, int H, int W, int Dq) {
    __shared__ float dg[2 * kVbRedT + 4];
    const int64_t row = blockIdx.x;  // (b*32 + o)*H + y
    const int y = (int)(row % H);
    const int64_t bo = row / H;
    const int u0 = (int)blockIdx.y * 2 * kVbRedT;
    const size_t HW = (size_t)H * W;
    const TG* gr = g + (size_t)bo * Dq * HW + (size_t)y * W;
    for (int i = threadIdx.x; i < 2 * kVbRedT + 4; i += kVbRedT) {
        const int v = u0 - 2 + i;
        const int dlo = max(1, -v), dhi = min(Dq - 2, W - 2 - v);
        float acc = 0.f;
#pragma unroll 8
        for (int d = dlo; d <= dhi; ++d) acc += ld_f32(gr + (size_t)d * HW + (v + d));
        dg[i] = acc;
    }
    __syncthreads();
    const int xl = 2 * (int)threadIdx.x, x = u0 + xl;
    if (x >= W) return;  // W even: x + 1 < W too
    const TG* gc = gr + x;
    const float2 g0 = ld2_f32(gc);
    const float2 gl = Dq >= 2 ? ld2_f32(gc + (size_t)(Dq - 1) * HW) : make_float2(0.f, 0.f);
    // column x: plain accumulation to plane x-3, snapshots at planes x-2 .. x+2 (k = 0..4);
    // column x+1: plain accumulation to plane x-2 (k = 0), snapshots at planes x-1 .. x+3 (k = 1..5)
    float M0 = 0.f, M1 = 0.f, snap0[5], snap1[5];
    const int e0 = min(x - 3, Dq - 2);
#pragma unroll 8
    for (int d = 1; d <= e0; ++d) {
        const float2 v = ld2_f32(gc + (size_t)d * HW);
        M0 += v.x;
        M1 += v.y;
    }
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        const int e = x + k - 2;
        if (e >= 1 && e <= Dq - 2) {
            const float2 v = ld2_f32(gc + (size_t)e * HW);
            if (k < 5) M0 += v.x;
            M1 += v.y;
        }
        if (k < 5) snap0[k] = M0;
        if (k > 0) snap1[k - 1] = M1;
    }
    const size_t NP = (size_t)B * kVbC * HW;
    float* out = planes + (size_t)row * W + x;
#pragma unroll
    for (int kd = 0; kd < 3; ++kd) {
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
            const int s = kx - kd;
            float a[2];
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                const int xc = x + c;
                const float m = c ? snap1[s + 2] : snap0[s + 2];
                const float last = (xc + s >= Dq - 1) ? (c ? gl.y : gl.x) : 0.f;
                const float h0 = c ? g0.y : g0.x;
                if (kd == 0) a[c] = m + last;
                else if (kd == 1) a[c] = (xc + s >= 0) ? (h0 + m) + last : 0.f;
                else a[c] = (xc + s >= 0 && Dq >= 2) ? h0 + m : 0.f;
            }
            *reinterpret_cast<float2*>(out + (size_t)(kd * 3 + kx) * NP) = make_float2(a[0], a[1]);
        }
    }
#pragma unroll
    for (int kd = 0; kd < 3; ++kd) {
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
            float zz[2];
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                const int t = kd - kx, v = x + c + t, xmax = W - 1 - (kx == 2 ? 1 : 0);
                float z = dg[xl + c + 2 + t];
                if ((kd == 1 || (kd == 2 && Dq >= 2)) && v >= 0 && v <= xmax) z += ld_f32(gr + v);
                const int vl = v + Dq - 1;
                if (kd <= 1 && Dq >= 2 && vl >= 0 && vl <= xmax) z += ld_f32(gr + (size_t)(Dq - 1) * HW + vl);
                const int dw = W - 1 - v;
                if (kx <= 1 && dw >= 1 && dw <= Dq - 2) z += ld_f32(gr + (size_t)dw * HW + (W - 1));
                zz[c] = z;
            }
            *reinterpret_cast<float2*>(out + (size_t)(9 + kd * 3 + kx) * NP) = make_float2(zz[0], zz[1]);
        }
    }
}

// ------------------------------------------------------------------------------------------
// 2. dfeat.  grid = (B*H, ceil(W / kVbTX), 2 halves), 128 threads: warp w owns channels 8w .. 8w+7, lane l the columns
// x0 + l + 32j (j = 0..3).  Per tap (kd, kx) the CTA stages the three rows y'-ky+1 of the 32 planes, shifted by
// 1 - kx (left half) or not at all (right half), and the 3 x 32 x 32 weights; the sum runs over (kd, kx, ky, o) in
// that order, one FMA chain per output.
// ------------------------------------------------------------------------------------------
// The weight dfeat contracts with: a weight of the features' type TF is widened exactly; an fp32 weight used with
// 16-bit features is first rounded to TF (RNE), as the 16-bit forward's pack and torch.autocast round it.
template <typename TF, typename TW>
__device__ __forceinline__ float vcb_weight(const TW* p) {
    if constexpr (std::is_same<TF, TW>::value || std::is_same<TF, float>::value) return ld_f32(p);
    else if constexpr (std::is_same<TF, __nv_bfloat16>::value) return __bfloat162float(__float2bfloat16_rn(__ldg(p)));
    else return __half2float(__float2half_rn(__ldg(p)));
}

template <typename TF, typename TW>
__global__ void __launch_bounds__(128) vcb_dfeat_kernel(const float* __restrict__ planes, const TW* __restrict__ weight,
                                                        TF* __restrict__ gL, TF* __restrict__ gR, int B, int H,
                                                        int W) {
    extern __shared__ __align__(16) float vsm[];
    float* sin = vsm;                       // [ky][o][kVbTX]
    float* sw = vsm + 3 * kVbC * kVbTX;     // [ky][o][c]
    const int h = blockIdx.z;
    TF* gout = h ? gR : gL;
    if (gout == nullptr) return;
    const int tid = threadIdx.x, lane = tid & 31, cg = tid >> 5;
    const int by = blockIdx.x, b = by / H, y = by - b * H;
    const int x0 = (int)blockIdx.y * kVbTX;
    const size_t HW = (size_t)H * W;
    float acc[8][4];
#pragma unroll
    for (int c = 0; c < 8; ++c)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[c][j] = 0.f;
    for (int kd = 0; kd < 3; ++kd) {
        for (int kx = 0; kx < 3; ++kx) {
            const int p = h * 9 + kd * 3 + kx;
            const int sh = h ? 0 : 1 - kx;
            const float* pl = planes + ((size_t)p * B + b) * kVbC * HW;
            __syncthreads();
            for (int i = tid; i < 3 * kVbC * kVbTX; i += 128) {
                const int xl = i % kVbTX, o = (i / kVbTX) % kVbC, ky = i / (kVbC * kVbTX);
                const int yy = y - ky + 1, xx = x0 + xl + sh;
                float v = 0.f;
                if (yy >= 0 && yy < H && xx >= 0 && xx < W) v = __ldg(pl + (size_t)o * HW + (size_t)yy * W + xx);
                sin[i] = v;
            }
            for (int i = tid; i < 3 * kVbC * kVbC; i += 128) {
                const int c = i % kVbC, o = (i / kVbC) % kVbC, ky = i / (kVbC * kVbC);
                sw[i] = vcb_weight<TF>(weight + (((size_t)o * 64 + h * kVbC + c) * 3 + kd) * 9 + ky * 3 + kx);
            }
            __syncthreads();
            for (int ky = 0; ky < 3; ++ky) {
#pragma unroll 4
                for (int o = 0; o < kVbC; ++o) {
                    const float* wr = sw + (ky * kVbC + o) * kVbC + cg * 8;
                    const float4 w0 = *reinterpret_cast<const float4*>(wr);
                    const float4 w1 = *reinterpret_cast<const float4*>(wr + 4);
                    const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
                    const float* ir = sin + (ky * kVbC + o) * kVbTX + lane;
                    float a[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j) a[j] = ir[32 * j];
#pragma unroll
                    for (int c = 0; c < 8; ++c)
#pragma unroll
                        for (int j = 0; j < 4; ++j) acc[c][j] = fmaf(wv[c], a[j], acc[c][j]);
                }
            }
        }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int x = x0 + lane + 32 * j;
        if (x >= W) continue;
#pragma unroll
        for (int c = 0; c < 8; ++c) st_from_f32(gout + ((size_t)b * kVbC + cg * 8 + c) * HW + (size_t)y * W + x, acc[c][j]);
    }
}

// ------------------------------------------------------------------------------------------
// 3. wgrad.  grid = (nchunks, 18 planes), kVwT threads: thread (ky = tid/64, og = (tid/8)%8, cg = tid%8) owns
// dW[o = 4og..4og+3][c = 4cg..4cg+3] of tap (kd, ky, kx) of the plane's half.  A chunk is rows_per_chunk consecutive
// image rows (b, y'); each row is swept in tiles of kVwTX positions staged position-major in shared memory
// (plane rows y'-ky+1 shifted like dfeat, features row y'); positions in order, one FMA chain per output.
// partial[p][chunk][ky][o][c].
// ------------------------------------------------------------------------------------------
template <typename TF>
__global__ void __launch_bounds__(kVwT) vcb_wgrad_kernel(const float* __restrict__ planes, const TF* __restrict__ L,
                                                         const TF* __restrict__ R, float* __restrict__ partial, int B,
                                                         int H, int W, int rows_per_chunk, int nchunks) {
    __shared__ __align__(16) float sin[3][kVwTX][kVwP];
    __shared__ __align__(16) float sf[kVwTX][kVwP];
    const int tid = threadIdx.x;
    const int p = blockIdx.y, h = p / 9, kx = p % 3;
    const int sh = h ? 0 : 1 - kx;
    const TF* F = h ? R : L;
    const int ky = tid >> 6, og = (tid >> 3) & 7, cg = tid & 7;
    const size_t HW = (size_t)H * W;
    const int nrows = B * H;
    const int r0 = (int)blockIdx.x * rows_per_chunk, r1 = min(nrows, r0 + rows_per_chunk);
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    for (int r = r0; r < r1; ++r) {
        const int b = r / H, y = r - b * H;
        const float* pl = planes + ((size_t)p * B + b) * kVbC * HW;
        const TF* fr = F + (size_t)b * kVbC * HW + (size_t)y * W;
        for (int x0 = 0; x0 < W; x0 += kVwTX) {
            __syncthreads();
            for (int i = tid; i < 3 * kVbC * kVwTX; i += kVwT) {
                const int xl = i % kVwTX, o = (i / kVwTX) % kVbC, k = i / (kVbC * kVwTX);
                const int yy = y - k + 1, xx = x0 + xl + sh;
                float v = 0.f;
                if (yy >= 0 && yy < H && xx >= 0 && xx < W) v = __ldg(pl + (size_t)o * HW + (size_t)yy * W + xx);
                sin[k][xl][o] = v;
            }
            for (int i = tid; i < kVbC * kVwTX; i += kVwT) {
                const int xl = i % kVwTX, c = i / kVwTX, x = x0 + xl;
                sf[xl][c] = x < W ? ld_f32(fr + (size_t)c * HW + x) : 0.f;
            }
            __syncthreads();
#pragma unroll 8
            for (int xl = 0; xl < kVwTX; ++xl) {
                const float4 a = *reinterpret_cast<const float4*>(&sin[ky][xl][4 * og]);
                const float4 f = *reinterpret_cast<const float4*>(&sf[xl][4 * cg]);
                const float av[4] = {a.x, a.y, a.z, a.w}, fv[4] = {f.x, f.y, f.z, f.w};
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], fv[j], acc[i][j]);
            }
        }
    }
    float* out = partial + (((size_t)p * nchunks + blockIdx.x) * 3 + ky) * (kVbC * kVbC);
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) out[(4 * og + i) * kVbC + 4 * cg + j] = acc[i][j];
}

// 4. finalize: one thread per element of dW [32][64][3][3][3]; the chunk partials are added in chunk order.
template <typename TW>
__global__ void __launch_bounds__(256) vcb_wgrad_finalize_kernel(const float* __restrict__ partial, TW* __restrict__ gW,
                                                                 int nchunks) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= kVbC * 64 * 27) return;
    const int kx = i % 3, ky = (i / 3) % 3, kd = (i / 9) % 3, ci = (i / 27) % 64, o = i / (27 * 64);
    const int h = ci / kVbC, c = ci - h * kVbC, p = h * 9 + kd * 3 + kx;
    const float* src = partial + ((size_t)p * nchunks * 3 + ky) * (kVbC * kVbC) + o * kVbC + c;
    float acc = 0.f;
    for (int ch = 0; ch < nchunks; ++ch) acc += src[(size_t)ch * 3 * kVbC * kVbC];
    st_from_f32(gW + i, acc);
}

inline size_t vcb_planes_bytes(int64_t B, int64_t H, int64_t W) {
    return (size_t)ceil_div((int64_t)kVbPlanes * B * kVbC * H * W * 4, 256) * 256;
}

static int vcb_check(const void* gout, const void* L, const void* R, const void* weight, int64_t B, int64_t C, int64_t H,
                     int64_t W, int64_t Dq) {
    if (!gout || !L || !R || !weight || B <= 0 || H <= 0 || W <= 0 || Dq <= 0) return AZ_ERR_BAD_ARG;
    if (C != kVbC) return AZ_ERR_BAD_ARG;  // PSMNet: 32 + 32 -> 32 channels, as the forward
    if (H * W >= (1ll << 31) || B * kVbC * H >= (1ll << 31) || ceil_div(W, kVbTX) > 65535) return AZ_ERR_BAD_ARG;
    return 0;
}

// TF: g, the features and their gradients; TW: the weight and dW (float, or TF when TF is 16-bit)
template <typename TF, typename TW>
int vcb_launch(const TF* gout, const TF* L, const TF* R, const TW* weight, TF* gL, TF* gR, TW* gW, void* workspace,
               int64_t B, int64_t H, int64_t W, int64_t Dq, cudaStream_t st) {
    if (!gL && !gR && !gW) return 0;
    if (!workspace) return AZ_ERR_BAD_ARG;
    float* planes = reinterpret_cast<float*>(workspace);
    if constexpr (!std::is_same<TF, float>::value) {
        if (W % 2 == 0 && (reinterpret_cast<uintptr_t>(gout) & 3u) == 0) {
            dim3 grid((unsigned)(B * kVbC * H), (unsigned)ceil_div(W, 2 * kVbRedT));
            vcb_reduce2_kernel<TF><<<grid, kVbRedT, 0, st>>>(gout, planes, (int)B, (int)H, (int)W, (int)Dq);
            AZ_LAUNCH_CHECK();
        } else {
            dim3 grid((unsigned)(B * kVbC * H), (unsigned)ceil_div(W, kVbRedT));
            vcb_reduce_kernel<TF><<<grid, kVbRedT, 0, st>>>(gout, planes, (int)B, (int)H, (int)W, (int)Dq);
            AZ_LAUNCH_CHECK();
        }
    } else {
        dim3 grid((unsigned)(B * kVbC * H), (unsigned)ceil_div(W, kVbRedT));
        vcb_reduce_kernel<TF><<<grid, kVbRedT, 0, st>>>(gout, planes, (int)B, (int)H, (int)W, (int)Dq);
        AZ_LAUNCH_CHECK();
    }
    if (gL || gR) {
        cudaError_t e = cudaFuncSetAttribute(vcb_dfeat_kernel<TF, TW>, cudaFuncAttributeMaxDynamicSharedMemorySize, kVbDfSmem);
        if (e != cudaSuccess) return (int)e;
        dim3 grid((unsigned)(B * H), (unsigned)ceil_div(W, kVbTX), 2);
        vcb_dfeat_kernel<TF, TW><<<grid, 128, kVbDfSmem, st>>>(planes, weight, gL, gR, (int)B, (int)H, (int)W);
        AZ_LAUNCH_CHECK();
    }
    if (gW) {
        const int rpc = (int)vcb_rows_per_chunk(B, H), nch = (int)vcb_nchunks(B, H);
        float* partial = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + vcb_planes_bytes(B, H, W));
        dim3 grid((unsigned)nch, kVbPlanes);
        vcb_wgrad_kernel<TF><<<grid, kVwT, 0, st>>>(planes, L, R, partial, (int)B, (int)H, (int)W, rpc, nch);
        AZ_LAUNCH_CHECK();
        vcb_wgrad_finalize_kernel<TW><<<(unsigned)ceil_div(kVbC * 64 * 27, 256), 256, 0, st>>>(partial, gW, nch);
        AZ_LAUNCH_CHECK();
    }
    return 0;
}

}  // namespace az

using namespace az;

extern "C" int64_t az_volume_conv0_bwd_workspace_bytes(int64_t B, int64_t H, int64_t W, int64_t Dq) {
    if (B <= 0 || H <= 0 || W <= 0 || Dq <= 0) return 0;
    return (int64_t)vcb_planes_bytes(B, H, W) + (int64_t)kVbPlanes * vcb_nchunks(B, H) * 3 * kVbC * kVbC * 4;
}

extern "C" int az_volume_conv0_bwd(const float* gout, const float* L, const float* R, const float* weight, float* gL,
                                   float* gR, float* gW, void* workspace, int64_t B, int64_t C, int64_t H, int64_t W,
                                   int64_t Dq, void* stream) {
    const int rc = vcb_check(gout, L, R, weight, B, C, H, W, Dq);
    if (rc != 0) return rc;
    return vcb_launch<float, float>(gout, L, R, weight, gL, gR, gW, workspace, B, H, W, Dq, (cudaStream_t)stream);
}

template <typename T>
static int vcb_launch16(const void* gout, const void* L, const void* R, const void* weight, void* gL, void* gR, void* gW,
                        void* workspace, int64_t B, int64_t H, int64_t W, int64_t Dq, int weight_dtype, cudaStream_t st) {
    const T* g = static_cast<const T*>(gout);
    const T* l = static_cast<const T*>(L);
    const T* r = static_cast<const T*>(R);
    if (weight_dtype == 0)
        return vcb_launch<T, float>(g, l, r, static_cast<const float*>(weight), static_cast<T*>(gL), static_cast<T*>(gR),
                                    static_cast<float*>(gW), workspace, B, H, W, Dq, st);
    return vcb_launch<T, T>(g, l, r, static_cast<const T*>(weight), static_cast<T*>(gL), static_cast<T*>(gR),
                            static_cast<T*>(gW), workspace, B, H, W, Dq, st);
}

extern "C" int az_volume_conv0_bwd_16(const void* gout, const void* L, const void* R, const void* weight, void* gL,
                                      void* gR, void* gW, void* workspace, int64_t B, int64_t C, int64_t H, int64_t W,
                                      int64_t Dq, int dtype, int weight_dtype, void* stream) {
    if ((dtype != AZ_DTYPE_BF16 && dtype != AZ_DTYPE_F16) || (weight_dtype != 0 && weight_dtype != dtype))
        return AZ_ERR_BAD_ARG;
    const int rc = vcb_check(gout, L, R, weight, B, C, H, W, Dq);
    if (rc != 0) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == AZ_DTYPE_BF16)
        return vcb_launch16<__nv_bfloat16>(gout, L, R, weight, gL, gR, gW, workspace, B, H, W, Dq, weight_dtype, st);
    return vcb_launch16<__half>(gout, L, R, weight, gL, gR, gW, workspace, B, H, W, Dq, weight_dtype, st);
}
