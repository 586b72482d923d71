// Image gradients of the fused reprojection losses (warp_reproj.cu, patch_loss_fold*.cu): d loss / d tgt and
// d loss / d src of reprojection.py:81-127 without the [B,C*ps*ps,H,W] unfolded / warped tensors.  DESIGN.md §4.14.
//
// Notation (one channel plane c, pixel (i,j), tap k = (ky,kx), p = (ps-1)/2):
//   r_k(i,j)   = Wu_k(i,j) - tgt[c, i+ky-p, j+kx-p]          (0 outside the image: Unfold's zero padding)
//   Wu_k(i,j)  = sum_{a,b} wy_a(i) wx_b(i,j) src[c, y0(i)+a+ky-p, x0(i,j)+b+kx-p]
//   rho_k(i,j) = s * m(i,j) * r_k(i,j),   s = gloss * 2 / (K * sum m),  K = C*ps*ps
// with the corner weights folded with the validity flags of the unfolded plane (make_axis: v0 / v1), exactly as the
// forward kernels form them.  Then
//   gtgt[c,y,x] = - sum_{ky,kx} rho_k(y+p-ky, x+p-kx)                          (a gather: reproj_gtgt_kernel)
//   gsrc[c,Y,X] = + sum rho_k(i,j) * wy_a(i) * wx_b(i,j) over y0(i)+a+ky-p = Y, x0(i,j)+b+kx-p = X
//                                                                           (a scatter: reproj_gsrc_kernel)
// The residuals are recomputed from tgt, src, disp and the mask; nothing of size K is stored.  Both kernels are
// deterministic: the gather sums in a fixed order, the scatter adds into 64-bit fixed-point words (integer addition
// is associative) as warp_bwd_img_kernel does, and every output element is stored exactly once.
#include <climits>

#include "common.cuh"

namespace az {

constexpr int kImgThreads = 256;
constexpr int kGsrcTile = 8192;  // gsrc columns per CTA: 64 KB of accumulators, three CTAs per SM

// Corner weights of the x axis of pixel (i,j), as the forward forms them (reproj_loss_kernel, fold_src).
struct XCorner {
    int x0;          // floor(xs) clamped to [-1, W-1]: outside that range both weights are 0
    float bx0, bx1;  // corner weights with the unfolded plane's validity folded in
};

__device__ __forceinline__ XCorner x_corner(const float* __restrict__ drow, const float* __restrict__ lin_x, float sign,
                                            int j, int W) {
    const Axis ax = make_axis(sample_pos(__ldg(lin_x + j), __fdiv_rn(sign * __ldg(drow + j), (float)W), (float)W), W);
    XCorner q;
    q.x0 = min(max(ax.i0, -1), W - 1);
    q.bx0 = ax.v0 ? ax.e : 0.f;
    q.bx1 = ax.v1 ? ax.w : 0.f;
    return q;
}

__device__ __forceinline__ float ld_or0(const float* __restrict__ row, bool rowok, int x, int W) {
    return (rowok && x >= 0 && x < W) ? __ldg(row + x) : 0.f;
}

// s = gloss * 2 / (K * sum m); the caller handles sum m == 0 (exact zeros)
__device__ __forceinline__ double grad_scale(const double* __restrict__ stats, const float* __restrict__ gloss, double K) {
    return (double)gloss[0] * 2.0 / (K * stats[1]);
}

// ------------------------------------------------------------------------------------------
// gtgt: one CTA per (256 output columns, output row y, b), one thread per column, channels in turn.  For tap row ky
// the contributing source row is i = y+p-ky; the corner parameters of its columns x-p .. x+p+255 are staged once per
// (c, ky) in shared memory, and each thread sums m * (Wu_k - tgt[y,x]) over kx in a fixed order (fp64 accumulator).
// grid = (nchunk * H, B), dynamic smem = (256 + 2p) * 12 bytes.
// ------------------------------------------------------------------------------------------
template <int PS>
__global__ void __launch_bounds__(kImgThreads) reproj_gtgt_kernel(
    const float* __restrict__ tgt, const float* __restrict__ src, const float* __restrict__ disp, float sign,
    const uint8_t* __restrict__ mask, const float* __restrict__ lin_x, const float* __restrict__ lin_y, int ps,
    const double* __restrict__ stats, const float* __restrict__ gloss, float* __restrict__ gtgt, int C, int H, int W,
    int nchunk) {
    extern __shared__ __align__(16) float smf[];
    const int n = PS > 0 ? PS : ps;
    const int p = (n - 1) >> 1;
    const int span = kImgThreads + 2 * p;
    int* Px0 = reinterpret_cast<int*>(smf);
    float* Pb0 = smf + span;
    float* Pb1 = smf + 2 * span;
    const int y = blockIdx.x / nchunk, X0 = (blockIdx.x - y * nchunk) * kImgThreads, b = blockIdx.y;
    const int x = X0 + threadIdx.x;
    const bool xin = x < W;
    const size_t HW = (size_t)H * W;
    const bool empty = stats[1] == 0.0;  // empty mask: the reference's image gradients are exactly zero
    const double s = empty ? 0.0 : grad_scale(stats, gloss, (double)C * n * n);
    const float* dplane = disp + (size_t)b * HW;
    for (int c = 0; c < C; ++c) {
        const size_t plane = ((size_t)b * C + c) * HW;
        const float* sp = src + plane;
        const float t = xin ? __ldg(tgt + plane + (size_t)y * W + x) : 0.f;
        double acc = 0.0;
        for (int ky = 0; ky < n && !empty; ++ky) {
            const int i = y + p - ky;
            if (i < 0 || i >= H) continue;  // CTA-uniform
            const Axis ay = make_axis(sample_pos(__ldg(lin_y + i), 0.0f, (float)H), H);
            const float ay0 = ay.v0 ? ay.e : 0.f, ay1 = ay.v1 ? ay.w : 0.f;
            const int r0 = ay.i0 + ky - p;  // image rows r0, r0+1 blended by tap row ky
            const bool ok0 = r0 >= 0 && r0 < H, ok1 = r0 + 1 >= 0 && r0 + 1 < H;
            const float* row0 = sp + (size_t)(ok0 ? r0 : 0) * W;
            const float* row1 = sp + (size_t)(ok1 ? r0 + 1 : 0) * W;
            __syncthreads();  // the previous tap row's parameters are consumed
            for (int q = threadIdx.x; q < span; q += kImgThreads) {
                const int j = X0 - p + q;
                int x0 = INT_MIN;  // INT_MIN: source pixel outside the image or not selected by the mask
                float b0 = 0.f, b1 = 0.f;
                if (j >= 0 && j < W && (mask == nullptr || mask[(size_t)b * HW + (size_t)i * W + j] != 0)) {
                    const XCorner xc = x_corner(dplane + (size_t)i * W, lin_x, sign, j, W);
                    x0 = xc.x0;
                    b0 = xc.bx0;
                    b1 = xc.bx1;
                }
                Px0[q] = x0;
                Pb0[q] = b0;
                Pb1[q] = b1;
            }
            __syncthreads();
            if (!xin) continue;
#pragma unroll
            for (int kx = 0; kx < n; ++kx) {
                const int q = threadIdx.x + 2 * p - kx;  // source column j = x+p-kx
                const int x0 = Px0[q];
                if (x0 == INT_MIN) continue;
                const int xa = x0 + kx - p;
                const float B0 = fmaf(ay1, ld_or0(row1, ok1, xa, W), ay0 * ld_or0(row0, ok0, xa, W));
                const float B1 = fmaf(ay1, ld_or0(row1, ok1, xa + 1, W), ay0 * ld_or0(row0, ok0, xa + 1, W));
                acc += (double)(fmaf(Pb1[q], B1, Pb0[q] * B0) - t);
            }
        }
        if (xin) gtgt[plane + (size_t)y * W + x] = empty ? 0.f : (float)(-s * acc);
    }
}

// ------------------------------------------------------------------------------------------
// gsrc: one CTA per (tile of <= kGsrcTile output columns, output row Y, b), channels in turn.  ys(i) grows by
// H/(H-1) > 1 per row, so for each (ky, a) at most one source row i has y0(i) = Y-a-ky+p: a table of <= 2*ps
// (i, wy) entries.  For each entry the threads walk the pixels j of row i, recompute the ps residuals of tap row ky
// (the blended source rows are Y-a and Y-a+1, the target row i+ky-p) and add rho * wy * wx_b to column
// x0+b+kx-p of a shared row of 64-bit fixed-point accumulators.  The fixed-point scale bounds the worst case --
// every contribution of the row landing on one column, |r| <= max|src| + max|tgt| over the rows read -- so it
// cannot overflow: at most 2*ps entries x W pixels x 2 (kx, b) pairs per column.  A non-finite value among those
// rows makes the output row NaN (fixed point cannot carry it).  The bound is 2 * the largest magnitude read.
// grid = (ntile * H, B), 256 threads, dynamic smem = tile * 8 + 2*ps * 16 bytes.
// ------------------------------------------------------------------------------------------
template <int PS>
__global__ void __launch_bounds__(kImgThreads, 2) reproj_gsrc_kernel(
    const float* __restrict__ tgt, const float* __restrict__ src, const float* __restrict__ disp, float sign,
    const uint8_t* __restrict__ mask, const float* __restrict__ lin_x, const float* __restrict__ lin_y, int ps,
    const double* __restrict__ stats, const float* __restrict__ gloss, float* __restrict__ gsrc, int C, int H, int W,
    int ntile) {
    extern __shared__ __align__(16) unsigned long long facc[];
    __shared__ float red[kImgThreads / 32];
    __shared__ int trow_lo, trow_hi;
    const int n = PS > 0 ? PS : ps;
    const int p = (n - 1) >> 1;
    const int Y = blockIdx.x / ntile, X0 = (blockIdx.x - Y * ntile) * kGsrcTile, b = blockIdx.y;
    const int XT = min(W - X0, kGsrcTile);
    const int tid = threadIdx.x;
    int* Ei = reinterpret_cast<int*>(facc + kGsrcTile);  // entry e = 2*ky + a: source row i, or -1
    float* Ewy = reinterpret_cast<float*>(Ei + 2 * n);    // wy_a(i)
    float* Ea0 = Ewy + 2 * n;                             // row weights of the blended source row
    float* Ea1 = Ea0 + 2 * n;
    const size_t HW = (size_t)H * W;
    const float* dplane = disp + (size_t)b * HW;
    const uint8_t* mplane = mask == nullptr ? nullptr : mask + (size_t)b * HW;

    for (int e = tid; e < 2 * n; e += kImgThreads) {
        const int ky = e >> 1, a = e & 1;
        const int y0 = Y - a - ky + p;
        int ii = -1;
        float wy = 0.f, a0 = 0.f, a1 = 0.f;
        for (int i = max(y0 - 1, 0); i <= min(y0 + 2, H - 1); ++i) {
            const Axis ay = make_axis(sample_pos(__ldg(lin_y + i), 0.0f, (float)H), H);
            const float w = a == 0 ? (ay.v0 ? ay.e : 0.f) : (ay.v1 ? ay.w : 0.f);
            if (ay.i0 == y0 && w != 0.f) {
                ii = i;
                wy = w;
                a0 = ay.v0 ? ay.e : 0.f;
                a1 = ay.v1 ? ay.w : 0.f;
            }
        }
        Ei[e] = ii;
        Ewy[e] = wy;
        Ea0[e] = a0;
        Ea1[e] = a1;
    }
    __syncthreads();
    if (tid == 0) {
        int lo = H, hi = -1;
        for (int e = 0; e < 2 * n; ++e)
            if (Ei[e] >= 0) {
                lo = min(lo, Ei[e] + (e >> 1) - p);
                hi = max(hi, Ei[e] + (e >> 1) - p);
            }
        trow_lo = max(lo, 0);
        trow_hi = min(hi, H - 1);
    }
    __syncthreads();
    const int tlo = trow_lo, thi = trow_hi;
    const bool empty = stats[1] == 0.0;
    const double s = empty ? 0.0 : grad_scale(stats, gloss, (double)C * n * n);

    for (int c = 0; c < C; ++c) {
        const size_t plane = ((size_t)b * C + c) * HW;
        const float* sp = src + plane;
        const float* tp = tgt + plane;
        float* orow = gsrc + plane + (size_t)Y * W + X0;
        // |r| <= 2m, m = the largest magnitude among src rows Y-1..Y+1 and the target rows the entries read
        float m = 0.f;
        bool bad = false;
        for (int r = max(Y - 1, 0); r <= min(Y + 1, H - 1); ++r)
            for (int xx = tid; xx < W; xx += kImgThreads) {
                const float v = fabsf(__ldg(sp + (size_t)r * W + xx));
                bad |= !(v <= 3.402823466e38f);
                m = fmaxf(m, v);
            }
        for (int r = tlo; r <= thi; ++r)
            for (int xx = tid; xx < W; xx += kImgThreads) {
                const float v = fabsf(__ldg(tp + (size_t)r * W + xx));
                bad |= !(v <= 3.402823466e38f);
                m = fmaxf(m, v);
            }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        __syncthreads();  // red[] and facc of the previous channel are consumed
        if ((tid & 31) == 0) red[tid >> 5] = m;
        bad = __syncthreads_or(bad) != 0;
        m = red[0];
#pragma unroll
        for (int k = 1; k < kImgThreads / 32; ++k) m = fmaxf(m, red[k]);
        if (empty || m == 0.f || bad) {  // exact zeros (also 0 * s: NaN for a non-finite gloss), or NaN
            const float fill = bad && !empty ? __int_as_float(0x7fc00000) : (empty ? 0.f : (float)(0.0 * s));
            for (int xx = tid; xx < XT; xx += kImgThreads) orow[xx] = fill;
            continue;
        }
        const double scale = ldexp(1.0, 61) / (2.0 * (double)m * 4.0 * (double)n * (double)W);
        for (int xx = tid; xx < XT; xx += kImgThreads) facc[xx] = 0ull;
        __syncthreads();
        for (int e = 0; e < 2 * n; ++e) {
            const int i = Ei[e];
            if (i < 0) continue;  // CTA-uniform
            const int ky = e >> 1, a = e & 1;
            const float wy = Ewy[e], ay0 = Ea0[e], ay1 = Ea1[e];
            const int r0 = Y - a;  // blended source rows r0, r0+1
            const bool ok0 = r0 >= 0, ok1 = r0 + 1 < H;
            const float* row0 = sp + (size_t)(ok0 ? r0 : 0) * W;
            const float* row1 = sp + (size_t)(ok1 ? r0 + 1 : 0) * W;
            const int ti = i + ky - p;
            const bool tok = ti >= 0 && ti < H;
            const float* trow = tp + (size_t)(tok ? ti : 0) * W;
            for (int j = tid; j < W; j += kImgThreads) {
                if (mplane != nullptr && mplane[(size_t)i * W + j] == 0) continue;
                const XCorner xc = x_corner(dplane + (size_t)i * W, lin_x, sign, j, W);
                const float w0 = wy * xc.bx0, w1 = wy * xc.bx1;
#pragma unroll
                for (int kx = 0; kx < n; ++kx) {
                    const int xa = xc.x0 + kx - p;
                    const float B0 = fmaf(ay1, ld_or0(row1, ok1, xa, W), ay0 * ld_or0(row0, ok0, xa, W));
                    const float B1 = fmaf(ay1, ld_or0(row1, ok1, xa + 1, W), ay0 * ld_or0(row0, ok0, xa + 1, W));
                    const float r = fmaf(xc.bx1, B1, xc.bx0 * B0) - ld_or0(trow, tok, j + kx - p, W);
                    const int u0 = xa - X0;
                    if (w0 != 0.f && u0 >= 0 && u0 < XT)
                        atomicAdd(&facc[u0], (unsigned long long)__double2ll_rn((double)(r * w0) * scale));
                    if (w1 != 0.f && u0 + 1 >= 0 && u0 + 1 < XT)
                        atomicAdd(&facc[u0 + 1], (unsigned long long)__double2ll_rn((double)(r * w1) * scale));
                }
            }
        }
        __syncthreads();
        const double out_scale = s / scale;
        for (int xx = tid; xx < XT; xx += kImgThreads) orow[xx] = (float)((double)(long long)facc[xx] * out_scale);
    }
}

template <int PS>
static int launch_img_bwd(const float* tgt, const float* src, const float* disp, float sign, const uint8_t* mask,
                          const float* lin_x, const float* lin_y, int ps, const double* stats, const float* gloss,
                          float* gtgt, float* gsrc, int B, int C, int H, int W, cudaStream_t st) {
    const int p = (ps - 1) / 2;
    const size_t smem_t = (size_t)(kImgThreads + 2 * p) * 12;
    const size_t smem_s = (size_t)kGsrcTile * 8 + (size_t)2 * ps * 16;
    if (smem_t > 220 * 1024 || smem_s > 220 * 1024) return AZ_ERR_BAD_ARG;
    if (gtgt != nullptr) {
        cudaError_t e = cudaFuncSetAttribute(reproj_gtgt_kernel<PS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)(220 * 1024));
        if (e != cudaSuccess) return (int)e;
        const int nchunk = (int)ceil_div(W, kImgThreads);
        dim3 grid((unsigned)(nchunk * H), (unsigned)B);
        reproj_gtgt_kernel<PS><<<grid, kImgThreads, smem_t, st>>>(tgt, src, disp, sign, mask, lin_x, lin_y, ps, stats,
                                                                 gloss, gtgt, C, H, W, nchunk);
        AZ_LAUNCH_CHECK();
    }
    if (gsrc != nullptr) {
        cudaError_t e = cudaFuncSetAttribute(reproj_gsrc_kernel<PS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)(220 * 1024));
        if (e != cudaSuccess) return (int)e;
        const int ntile = (int)ceil_div(W, kGsrcTile);
        dim3 grid((unsigned)(ntile * H), (unsigned)B);
        reproj_gsrc_kernel<PS><<<grid, kImgThreads, smem_s, st>>>(tgt, src, disp, sign, mask, lin_x, lin_y, ps, stats,
                                                                 gloss, gsrc, C, H, W, ntile);
        AZ_LAUNCH_CHECK();
    }
    return 0;
}

}  // namespace az

using namespace az;

extern "C" int az_reproj_loss_img_bwd(const float* tgt, const float* src, const float* disp, float sign,
                                      const uint8_t* mask, const float* lin_x, const float* lin_y, int64_t ps,
                                      const double* stats, const float* gloss, float* gtgt, float* gsrc, int64_t B,
                                      int64_t C, int64_t H, int64_t W, void* stream) {
    if (!gtgt && !gsrc) return 0;
    if (!tgt || !src || !disp || !lin_x || !lin_y || !stats || !gloss) return AZ_ERR_BAD_ARG;
    if (B <= 0 || C <= 0 || H <= 0 || W <= 0 || ps < 1 || (ps % 2) == 0) return AZ_ERR_BAD_ARG;
    if (B > 65535 || H * W >= (1ll << 31) || ps > 4095) return AZ_ERR_BAD_ARG;  // larger ps: no shared-memory plan
    cudaStream_t st = (cudaStream_t)stream;
#define AZ_IMG_BWD(N)                                                                                                 \
    launch_img_bwd<N>(tgt, src, disp, sign, mask, lin_x, lin_y, (int)ps, stats, gloss, gtgt, gsrc, (int)B, (int)C, \
                      (int)H, (int)W, st)
    switch (ps) {
        case 1: return AZ_IMG_BWD(1);
        case 3: return AZ_IMG_BWD(3);
        case 5: return AZ_IMG_BWD(5);
        case 7: return AZ_IMG_BWD(7);
        case 9: return AZ_IMG_BWD(9);
        case 11: return AZ_IMG_BWD(11);
        case 13: return AZ_IMG_BWD(13);
        default: return AZ_IMG_BWD(0);
    }
#undef AZ_IMG_BWD
}
