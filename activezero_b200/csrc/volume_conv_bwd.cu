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
#include "common.cuh"

namespace az {

constexpr int kVbC = 32;           // feature channels per half (PSMNet)
constexpr int kVbPlanes = 18;      // A[kd,kx] (0..8), Z[kd,kx] (9..17)
constexpr int kVbRedT = 128;       // reduce: columns per CTA
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
__global__ void __launch_bounds__(kVbRedT) vcb_reduce_kernel(const float* __restrict__ g, float* __restrict__ planes,
                                                             int B, int H, int W, int Dq) {
    __shared__ float dg[kVbRedT + 4];
    const int64_t row = blockIdx.x;  // (b*32 + o)*H + y
    const int y = (int)(row % H);
    const int64_t bo = row / H;
    const int u0 = (int)blockIdx.y * kVbRedT;
    const size_t HW = (size_t)H * W;
    const float* gr = g + (size_t)bo * Dq * HW + (size_t)y * W;  // g[b,o,0,y,0]
    for (int i = threadIdx.x; i < kVbRedT + 4; i += kVbRedT) {
        const int v = u0 - 2 + i;
        const int dlo = max(1, -v), dhi = min(Dq - 2, W - 2 - v);
        float acc = 0.f;
#pragma unroll 8
        for (int d = dlo; d <= dhi; ++d) acc += __ldg(gr + (size_t)d * HW + (v + d));
        dg[i] = acc;
    }
    __syncthreads();
    const int x = u0 + (int)threadIdx.x;
    if (x >= W) return;
    const float* gc = gr + x;
    const float g0 = __ldg(gc);
    const float gl = Dq >= 2 ? __ldg(gc + (size_t)(Dq - 1) * HW) : 0.f;
    float M = 0.f, snap[5];
    const int e0 = min(x - 3, Dq - 2);
#pragma unroll 8
    for (int d = 1; d <= e0; ++d) M += __ldg(gc + (size_t)d * HW);
#pragma unroll
    for (int k = 0; k < 5; ++k) {
        const int e = x + k - 2;
        if (e >= 1 && e <= Dq - 2) M += __ldg(gc + (size_t)e * HW);
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
            if ((kd == 1 || (kd == 2 && Dq >= 2)) && v >= 0 && v <= xmax) z += __ldg(gr + v);
            const int vl = v + Dq - 1;
            if (kd <= 1 && Dq >= 2 && vl >= 0 && vl <= xmax) z += __ldg(gr + (size_t)(Dq - 1) * HW + vl);
            const int dw = W - 1 - v;
            if (kx <= 1 && dw >= 1 && dw <= Dq - 2) z += __ldg(gr + (size_t)dw * HW + (W - 1));
            out[(size_t)(9 + kd * 3 + kx) * NP] = z;
        }
    }
}

// ------------------------------------------------------------------------------------------
// 2. dfeat.  grid = (B*H, ceil(W / kVbTX), 2 halves), 128 threads: warp w owns channels 8w .. 8w+7, lane l the columns
// x0 + l + 32j (j = 0..3).  Per tap (kd, kx) the CTA stages the three rows y'-ky+1 of the 32 planes, shifted by
// 1 - kx (left half) or not at all (right half), and the 3 x 32 x 32 weights; the sum runs over (kd, kx, ky, o) in
// that order, one FMA chain per output.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) vcb_dfeat_kernel(const float* __restrict__ planes, const float* __restrict__ weight,
                                                        float* __restrict__ gL, float* __restrict__ gR, int B, int H,
                                                        int W) {
    extern __shared__ __align__(16) float vsm[];
    float* sin = vsm;                       // [ky][o][kVbTX]
    float* sw = vsm + 3 * kVbC * kVbTX;     // [ky][o][c]
    const int h = blockIdx.z;
    float* gout = h ? gR : gL;
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
                sw[i] = __ldg(weight + (((size_t)o * 64 + h * kVbC + c) * 3 + kd) * 9 + ky * 3 + kx);
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
        for (int c = 0; c < 8; ++c) gout[((size_t)b * kVbC + cg * 8 + c) * HW + (size_t)y * W + x] = acc[c][j];
    }
}

// ------------------------------------------------------------------------------------------
// 3. wgrad.  grid = (nchunks, 18 planes), kVwT threads: thread (ky = tid/64, og = (tid/8)%8, cg = tid%8) owns
// dW[o = 4og..4og+3][c = 4cg..4cg+3] of tap (kd, ky, kx) of the plane's half.  A chunk is rows_per_chunk consecutive
// image rows (b, y'); each row is swept in tiles of kVwTX positions staged position-major in shared memory
// (plane rows y'-ky+1 shifted like dfeat, features row y'); positions in order, one FMA chain per output.
// partial[p][chunk][ky][o][c].
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kVwT) vcb_wgrad_kernel(const float* __restrict__ planes, const float* __restrict__ L,
                                                         const float* __restrict__ R, float* __restrict__ partial, int B,
                                                         int H, int W, int rows_per_chunk, int nchunks) {
    __shared__ __align__(16) float sin[3][kVwTX][kVwP];
    __shared__ __align__(16) float sf[kVwTX][kVwP];
    const int tid = threadIdx.x;
    const int p = blockIdx.y, h = p / 9, kx = p % 3;
    const int sh = h ? 0 : 1 - kx;
    const float* F = h ? R : L;
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
        const float* fr = F + (size_t)b * kVbC * HW + (size_t)y * W;
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
                sf[xl][c] = x < W ? __ldg(fr + (size_t)c * HW + x) : 0.f;
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
__global__ void __launch_bounds__(256) vcb_wgrad_finalize_kernel(const float* __restrict__ partial, float* __restrict__ gW,
                                                                 int nchunks) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= kVbC * 64 * 27) return;
    const int kx = i % 3, ky = (i / 3) % 3, kd = (i / 9) % 3, ci = (i / 27) % 64, o = i / (27 * 64);
    const int h = ci / kVbC, c = ci - h * kVbC, p = h * 9 + kd * 3 + kx;
    const float* src = partial + ((size_t)p * nchunks * 3 + ky) * (kVbC * kVbC) + o * kVbC + c;
    float acc = 0.f;
    for (int ch = 0; ch < nchunks; ++ch) acc += src[(size_t)ch * 3 * kVbC * kVbC];
    gW[i] = acc;
}

inline size_t vcb_planes_bytes(int64_t B, int64_t H, int64_t W) {
    return (size_t)ceil_div((int64_t)kVbPlanes * B * kVbC * H * W * 4, 256) * 256;
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
    if (!gout || !L || !R || !weight || B <= 0 || H <= 0 || W <= 0 || Dq <= 0) return AZ_ERR_BAD_ARG;
    if (C != kVbC) return AZ_ERR_BAD_ARG;  // PSMNet: 32 + 32 -> 32 channels, as the forward
    if (H * W >= (1ll << 31) || B * kVbC * H >= (1ll << 31) || ceil_div(W, kVbTX) > 65535) return AZ_ERR_BAD_ARG;
    if (!gL && !gR && !gW) return 0;
    if (!workspace) return AZ_ERR_BAD_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    float* planes = reinterpret_cast<float*>(workspace);
    {
        dim3 grid((unsigned)(B * kVbC * H), (unsigned)ceil_div(W, kVbRedT));
        vcb_reduce_kernel<<<grid, kVbRedT, 0, st>>>(gout, planes, (int)B, (int)H, (int)W, (int)Dq);
        AZ_LAUNCH_CHECK();
    }
    if (gL || gR) {
        cudaError_t e = cudaFuncSetAttribute(vcb_dfeat_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kVbDfSmem);
        if (e != cudaSuccess) return (int)e;
        dim3 grid((unsigned)(B * H), (unsigned)ceil_div(W, kVbTX), 2);
        vcb_dfeat_kernel<<<grid, 128, kVbDfSmem, st>>>(planes, weight, gL, gR, (int)B, (int)H, (int)W);
        AZ_LAUNCH_CHECK();
    }
    if (gW) {
        const int rpc = (int)vcb_rows_per_chunk(B, H), nch = (int)vcb_nchunks(B, H);
        float* partial = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + vcb_planes_bytes(B, H, W));
        dim3 grid((unsigned)nch, kVbPlanes);
        vcb_wgrad_kernel<<<grid, kVwT, 0, st>>>(planes, L, R, partial, (int)B, (int)H, (int)W, rpc, nch);
        AZ_LAUNCH_CHECK();
        vcb_wgrad_finalize_kernel<<<(unsigned)ceil_div(kVbC * 64 * 27, 256), 256, 0, st>>>(partial, gW, nch);
        AZ_LAUNCH_CHECK();
    }
    return 0;
}
