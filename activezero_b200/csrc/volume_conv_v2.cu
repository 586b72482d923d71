// First convolution of the 3-D aggregation on the IMPLICIT concat volume, second form (round 2).
// (SURVEY.md §8f rank 2; /root/reference/nets/psmnet/psmnet.py:151-168, psmnet_submodule.py:44-56.)
//
// Why a second form.  volume_conv.cu gathers one 33 KB operand slab and re-reads 24 KB of weights per (kd, ky) of every
// 128-position tile: 516 KB of L2 traffic for 14 MFLOP, which bounds it at 1.3-1.5 ms per pair whatever the gather costs.
// This kernel removes that traffic with three observations:
//
//  1. SHIFTED OUTPUT COORDINATES.  Write the output column as x = xt + d.  The tap (kd, ky, kx) of out[d][y][xt + d] reads
//     the volume at x' = xt + d + kx - 1, d' = d + kd - 1, and
//        left half :  L[c][y'][xt + d + kx - 1]         -- the left row, shifted by d
//        right half:  R[c][y'][x' - d'] = R[c][y'][xt + kx - kd]   -- INDEPENDENT OF d
//        mask      :  x' >= d'  <=>  xt + kx >= kd       -- INDEPENDENT OF d
//     so the right half's contribution Q_kd[xt] is computed ONCE per (y, xt) for all Dq planes (three small GEMMs, one per
//     kd, because the first and the last plane lack one kd), and only the left half (K = 27 x 32) is a per-plane GEMM:
//     half of the FLOPs of the convolution are gone, which no convolution on the materialised volume can do.
//  2. FEATURE-STATIONARY.  In the no-swizzle K-major operand layout (8 rows x 16 bytes per core matrix) a 4-channel
//     chunk is linear in the row, so the A operand of plane d and tap kx is the SAME staged left rows read from a start
//     address (d + kx) x 16 bytes further: the three left rows (3 x 8 chunks x 184 positions x 16 B = 71 KB) and all 27
//     left-half weight blocks (108 KB) stay in shared memory for the whole CTA; the main loop issues tcgen05.mma and
//     nothing else -- no gather, no weight streaming.
//  3. The masks that remain are tiny and fixed: the mask xt + kx >= kd only bites in the rows xt = -2 .. 1 of the first
//     tile (the right half gets it for free from its zero prefix; the left half's 8 (row, tap) cases per plane are
//     tabulated on the CUDA cores before the main loop), and the volume's zero padding at x' = W only touches output
//     column W - 1 through the kx = 2 taps of the right half (tabulated the same way).  Columns x <= d - 3 see no
//     unmasked tap at all and are the epilogue of zero.
//
// CTA = one (b, y, tile of 128 shifted columns), all Dq planes.  Warps 0-3 are the epilogue (one TMEM lane = one output
// row each), warps 4-7 issue the MMAs (planes round-robin); accumulators of 8 planes live in tensor memory (8 x 32 columns, full / empty
// mbarriers), Q_0..2 in 96 more.  TF32 operands (cvt.rna at staging), fp32 accumulation, epilogue = optional
// scale / shift (eval-mode BatchNorm) and ReLU, NCDHW stores.
#include "common.cuh"

namespace az {

constexpr int kV2Issuers = 3;               // three issuing threads keep up with N = 96 (36 MMAs per plane)
constexpr int kV2Threads = 256 + 32 * kV2Issuers;  // warps 0-3 / 4-7: epilogue of the even / odd planes, then the issuers
constexpr int kV2M = 128, kV2N = 32, kV2C = 32;
constexpr int kV2RP = 184;                 // staged left positions: 128 + (Dq - 1) + 2 <= 184  =>  Dq <= 55
constexpr int kV2RQ = 136;                 // staged right positions: 128 + 2 + 2
constexpr int kV2MaxDq = 55;
constexpr int kV2MT = 126;                 // output columns per tile: 128 operand rows serve the three kx taps of 126
constexpr int kV2Slots = 4;                // accumulator slots in tensor memory (96 columns each: the three kx blocks)
constexpr int kV2CacheBytes = 3 * 8 * kV2RP * 16;   // 70 656
constexpr int kV2WBytes = 27 * 4096;                // 110 592: one half (32 channels) of every tap
constexpr int kV2ClFloats = kV2MaxDq * 4 * 32, kV2CrFloats = kV2MaxDq * 32;
constexpr int kV2Smem = kV2CacheBytes + kV2WBytes + (kV2ClFloats + kV2CrFloats) * 4;

__device__ __forceinline__ uint64_t v2_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    // cute::UMMA::SmemDescriptor: start address [0,14), leading byte offset [16,30), stride byte offset [32,46)
    // (all >> 4), version 1 at [46,48), layout type 0 (no swizzle)
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46);
}
// c_format F32, a/b TF32, both K-major, M = 128; N = 32 (right-half terms) or 96 (left half: the three kx taps of a
// (kd, ky) side by side -- in the no-swizzle layout tap kx is the same operand rows one row further, so the accumulator
// block kx of operand row u belongs to output row u - kx and the three blocks are summed with a row shift in the
// epilogue: the A operand is read once per 48 cycles of tensor-core math instead of once per 16)
constexpr uint32_t kV2Idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(kV2N >> 3) << 17) | ((uint32_t)(kV2M >> 4) << 24);
constexpr uint32_t kV2Idesc96 = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(96 >> 3) << 17) | ((uint32_t)(kV2M >> 4) << 24);

__device__ __forceinline__ float v2_tf32(float x) {
    uint32_t u;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
    return __uint_as_float(u);
}
__device__ __forceinline__ void v2_mma(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t accumulate, uint32_t idesc = kV2Idesc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, {%5, %6, %7, %8}, p;\n\t}"
        ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate), "r"(0), "r"(0), "r"(0), "r"(0)
        : "memory");
}
// wait with back-off: the issuing threads share their SM sub-partitions with the epilogue warps, and a tight try_wait
// loop (it returns at once when the phase is not complete) took half of their issue slots (60 M spins per launch)
__device__ __forceinline__ void v2_wait_sleep(uint64_t* bar, uint32_t parity) {
    const uint32_t a = smem_u32(bar);
    for (;;) {
        uint32_t ok;
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok) : "r"(a), "r"(parity) : "memory");
        if (ok) break;
        __nanosleep(128);
    }
}
__device__ __forceinline__ void v2_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void v2_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void v2_ld32(uint32_t taddr, uint32_t (&v)[32]) {
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
}

// float index of element (n, c) inside one half-tap block (4 KB) of the packed weights: [j = c/8][kc = (c/4)&1][ng][r][e]
__device__ __forceinline__ int v2_widx(int n, int c) {
    return (c & 3) + 4 * (n & 7) + 32 * (n >> 3) + 128 * ((c >> 2) & 1) + 256 * (c >> 3);
}

// sum_c w[c][n] * a[c] over the 32 channels of one half-tap block: both operands are 16-byte quads over c % 4
// (weights: [j = c/8][kc][ng][r][e], staged rows: [chunk c/4][row][4]); `chunk_stride` floats between chunks of `a`
template <int KC_STRIDE, int J_STRIDE>
__device__ __forceinline__ float v2_dot32(const float* __restrict__ wt, int n, const float* __restrict__ a, int chunk_stride) {
    const float* wn = wt + 4 * (n & 7) + 32 * (n >> 3);
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;  // four chains of 8 instead of one of 32 dependent FMAs
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const float4 w4 = *reinterpret_cast<const float4*>(wn + KC_STRIDE * (q & 1) + J_STRIDE * (q >> 1));
        const float4 a4 = *reinterpret_cast<const float4*>(a + (size_t)q * chunk_stride);
        a0 = fmaf(w4.x, a4.x, a0);
        a1 = fmaf(w4.y, a4.y, a1);
        a2 = fmaf(w4.z, a4.z, a2);
        a3 = fmaf(w4.w, a4.w, a3);
    }
    return (a0 + a1) + (a2 + a3);
}

// Stage three feature rows (y-1, y, y+1) of `src` in the operand layout: cache[ky][chunk kq][row][4 channels], row r
// holding image column col0 + r (zero outside the image / outside the rows), rounded to TF32 (16-bit features are
// widened first, which TF32 holds exactly).
template <typename T>
__device__ __forceinline__ void v2_stage_rows(float* __restrict__ cache, const T* __restrict__ src, int b, int y, int H,
                                              int W, int col0, int nrows) {
    const size_t HW = (size_t)H * W;
    for (int it = threadIdx.x; it < 3 * 8 * nrows; it += kV2Threads) {
        const int r = it % nrows, kq = (it / nrows) & 7, ky = it / (8 * nrows);
        const int yp = y + ky - 1, col = col0 + r;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (yp >= 0 && yp < H && col >= 0 && col < W) {
            const T* p = src + ((size_t)b * kV2C + 4 * kq) * HW + (size_t)yp * W + col;
            v.x = v2_tf32(ld_f32(p));
            v.y = v2_tf32(ld_f32(p + HW));
            v.z = v2_tf32(ld_f32(p + 2 * HW));
            v.w = v2_tf32(ld_f32(p + 3 * HW));
        }
        reinterpret_cast<float4*>(cache)[(size_t)(ky * 8 + kq) * nrows + r] = v;
    }
}
// Weights reach shared memory by bulk async copies (TMA) issued by one thread while the other threads stage the
// feature rows: the right half of the 27 tap blocks (4 KB each, tap-major) for phase 1, the left half in its N = 96
// order (second part of the packed buffer, 12 KB per (kd, ky)) for phase 3.
__device__ __forceinline__ void v2_copy_weights_right(float* ws, const float* __restrict__ wpacked, uint64_t* bar) {
    mbar_expect_tx(bar, 27u * 4096u);
    for (int tap = 0; tap < 27; ++tap) bulk_g2s(ws + tap * 1024, wpacked + (size_t)tap * 2048 + 1024, 4096u, bar);
}
__device__ __forceinline__ void v2_copy_weights_left96(float* ws, const float* __restrict__ wpacked, uint64_t* bar) {
    mbar_expect_tx(bar, 9u * 12288u);
    for (int k = 0; k < 9; ++k) bulk_g2s(ws + k * 3072, wpacked + (size_t)27 * 2048 + (size_t)k * 3072, 12288u, bar);
}

// T = the features' and the output's element type: float, or bf16 / fp16 (torch.autocast; the epilogue stays fp32 and
// rounds once at the store)
template <typename T>
__global__ void __launch_bounds__(kV2Threads, 1) volume_conv0_v2_kernel(const T* __restrict__ L, const T* __restrict__ R,
                                                                       const float* __restrict__ wpacked,
                                                                       const float* __restrict__ scale,
                                                                       const float* __restrict__ shift, T* __restrict__ out,
                                                                       int B, int H, int W, int Dq, int relu) {
    extern __shared__ __align__(128) unsigned char vsm[];
    __shared__ __align__(8) uint64_t bar_q, bar_w, full[kV2Slots], empty[kV2Slots];
    __shared__ uint32_t tmem_base_s;
    __shared__ float2 ss[32];              // eval-mode BatchNorm (scale, shift) per output channel, or (1, 0)
    __shared__ float xch[2][2][4][3][32];  // [group][plane parity within the group][warp][block][n]  // kx = 1 / 2 blocks of a warp's first two rows, for the previous warp's last rows
    float* cache = reinterpret_cast<float*>(vsm);
    float* ws = reinterpret_cast<float*>(vsm + kV2CacheBytes);
    float* Cl = reinterpret_cast<float*>(vsm + kV2CacheBytes + kV2WBytes);  // [Dq][4][32]
    float* Cr = Cl + kV2ClFloats;                                          // [Dq][32]
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int xt0 = -2 + kV2MT * (int)blockIdx.x;  // first shifted column of the tile
    const int y = blockIdx.y, b = blockIdx.z;
    const size_t HW = (size_t)H * W;
    const uint32_t sbase = smem_u32(vsm), wbase = sbase + kV2CacheBytes;

    if (tid < 32) ss[tid] = scale != nullptr ? make_float2(__ldg(scale + tid), __ldg(shift + tid)) : make_float2(1.f, 0.f);
    if (tid == 0) {
        mbar_init(&bar_q, 1);
        mbar_init(&bar_w, 1);
        for (int s = 0; s < kV2Slots; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 4);
        }
        mbar_fence_init();
        v2_copy_weights_right(ws, wpacked, &bar_w);  // overlaps the staging of the right rows
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    // ---- phase 1: right half.  Q_kd[m][n] = sum_{ky, kx, c} Wr[kd,ky,kx][c][n] * R[c][y'][xt0 + m + kx - kd]
    v2_stage_rows(cache, R, b, y, H, W, xt0 - 2, kV2RQ);  // row r <-> column xt0 - 2 + r;  operand row = m + kx - kd + 2
    mbar_wait(&bar_w, 0);
    fence_async_smem();
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = tmem_base_s;
    if (tid == 8 * 32) {
        for (int kd = 0; kd < 3; ++kd) {
            uint32_t acc = 0;
            for (int ky = 0; ky < 3; ++ky) {
                const int yp = y + ky - 1;
                if (yp < 0 || yp >= H) continue;
                for (int kx = 0; kx < 3; ++kx) {
                    const int tap = (kd * 3 + ky) * 3 + kx;
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const uint64_t da = v2_desc(sbase + (uint32_t)(((ky * 8 + 2 * j) * kV2RQ + (kx - kd + 2)) * 16), kV2RQ * 16, 128);
                        const uint64_t db = v2_desc(wbase + (uint32_t)(tap * 4096 + j * 1024), 512, 128);
                        v2_mma(tmem + 32 * kd, da, db, acc);
                        acc = 1;
                    }
                }
            }
        }
        v2_commit(&bar_q);
    }
    // right-border table (CUDA cores, while the tensor core computes Q): the volume is zero at x' = W, but the shifted right
    // operand holds R[W - d'] there -- only output column x = W - 1 sees it, through the kx = 2 taps.
    //   Cr[d][n] = sum_{kd valid, d' >= 1} sum_{ky valid} sum_c Wr[kd,ky,2][c][n] * R[c][y'][W - d']
    for (int o = tid; o < Dq * 32; o += kV2Threads) {
        const int d = o >> 5, n = o & 31;
        const int mstar = W - 1 - d - xt0;  // the tile row of output column W - 1 at plane d
        float acc = 0.f;
        if (mstar >= 0 && mstar < kV2MT) {
            for (int kd = 0; kd < 3; ++kd) {
                const int dp = d + kd - 1;
                if (dp < 1 || dp >= Dq) continue;
                const int row = mstar + 2 - kd + 2;  // operand row of tap kx = 2: column W - dp
                for (int ky = 0; ky < 3; ++ky) {
                    const int yp = y + ky - 1;
                    if (yp < 0 || yp >= H) continue;
                    acc += v2_dot32<128, 256>(ws + ((kd * 3 + ky) * 3 + 2) * 1024, n, cache + ((size_t)(ky * 8) * kV2RQ + row) * 4, kV2RQ * 4);
                }
            }
        }
        Cr[o] = acc;
    }
    mbar_wait(&bar_q, 0);  // Q complete: the staged right rows and weights may be overwritten
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    __syncthreads();
    // ---- phase 2: left half operands.  Operand row of (m, d, kx) = m + d + kx  <->  column xt0 - 1 + row = x + kx - 1
    if (tid == 0) v2_copy_weights_left96(ws, wpacked, &bar_w);  // the right-half weights are dead (Q is complete)
    v2_stage_rows(cache, L, b, y, H, W, xt0 - 1, kV2RP);
    mbar_wait(&bar_w, 1);
    fence_async_smem();
    __syncthreads();
    // left-mask table for the rows xt = -2 .. 1 of the first tile (mask xt + kx >= kd):
    //   rows 0, 1 (xt = -2, -1): the FULL left contribution (allowed taps only) -- replaces the accumulator
    //   rows 2, 3 (xt =  0,  1): the contribution of the masked taps             -- subtracted from the accumulator
    if (blockIdx.x == 0) {
        for (int o = tid; o < Dq * 4 * 32; o += kV2Threads) {
            const int n = o & 31, mrow = (o >> 5) & 3, d = o >> 7;
            const int xt = mrow - 2;
            float acc = 0.f;
            for (int kd = 0; kd < 3; ++kd) {
                const int dp = d + kd - 1;
                if (dp < 0 || dp >= Dq) continue;
                for (int kx = 0; kx < 3; ++kx) {
                    const bool allowed = xt + kx >= kd;
                    if ((xt < 0) != allowed) continue;  // xt < 0: sum the allowed taps; xt >= 0: sum the masked ones
                    const int row = mrow + d + kx;
                    for (int ky = 0; ky < 3; ++ky) {
                        const int yp = y + ky - 1;
                        if (yp < 0 || yp >= H) continue;
                        acc += v2_dot32<384, 768>(ws + (kd * 3 + ky) * 3072 + kx * 128, n, cache + ((size_t)(ky * 8) * kV2RP + row) * 4, kV2RP * 4);
                    }
                }
            }
            Cl[o] = acc;
        }
    }
    __syncthreads();

    // ---- phase 3: per-plane left-half GEMM (warp 4) and epilogue (warps 0-3), 8 accumulator slots in tensor memory
    if (warp >= 8) {
        // Four issuing threads, planes round-robin: one thread needs ~15 instructions per MMA (descriptor assembly on
        // the uniform datapath, elect, predicate) and cannot keep the tensor core busy alone (measured: 8 k cycles per
        // plane against 3.5 k of tensor-core time); accumulators are per plane, so the issuers are independent.
        if (lane == 0) {
            const uint64_t da0 = v2_desc(sbase, kV2RP * 16, 128), db0 = v2_desc(wbase, 1536, 128);
            for (int d = warp - 8; d < Dq; d += kV2Issuers) {
                const int s = d & (kV2Slots - 1);
                if (d >= kV2Slots) v2_wait_sleep(&empty[s], (uint32_t)(((d >> 2) - 1) & 1));
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t dst = tmem + 96 + 96 * s;
                uint32_t acc = 0;
                // descriptors differ from a base only in their start-address field (units of 16 bytes, no carry out
                // of the field: shared memory is < 256 KB): one 64-bit add per operand per MMA
                for (int kd = 0; kd < 3; ++kd) {
                    const int dp = d + kd - 1;
                    if (dp < 0 || dp >= Dq) continue;
                    for (int ky = 0; ky < 3; ++ky) {
                        const int yp = y + ky - 1;
                        if (yp < 0 || yp >= H) continue;
                        const uint64_t boff = (uint64_t)(((kd * 3 + ky) * 12288) >> 4);
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            const uint64_t da = da0 + (uint64_t)((ky * 8 + 2 * j) * kV2RP + d);
                            const uint64_t db = db0 + boff + (uint64_t)(j * 192);
                            v2_mma(dst, da, db, acc, kV2Idesc96);
                            acc = 1;
                        }
                    }
                }
                v2_commit(&full[s]);
            }
        }
    } else {
        const int grp = warp >> 2, wq = warp & 3;  // a warp reads the TMEM lanes 32 * (warp % 4) .. + 31
        const int m = tid & 127;                   // tile row = TMEM lane
        const uint32_t lane_base = tmem + ((uint32_t)(32 * wq) << 16);
        // Q_0 + Q_1 + Q_2 stays in registers; the first / last plane (no kd = 0 / kd = 2) re-read the missing term
        float qs[32];
        {
            uint32_t v[32];
            v2_ld32(lane_base + 0, v);
#pragma unroll
            for (int n = 0; n < 32; ++n) qs[n] = __uint_as_float(v[n]);
            v2_ld32(lane_base + 32, v);
#pragma unroll
            for (int n = 0; n < 32; ++n) qs[n] += __uint_as_float(v[n]);
            v2_ld32(lane_base + 64, v);
#pragma unroll
            for (int n = 0; n < 32; ++n) qs[n] += __uint_as_float(v[n]);
        }
        const size_t cstride = (size_t)Dq * HW;
        for (int d = grp; d < Dq; d += 2) {
            const int s = d & (kV2Slots - 1);
            mbar_wait(&full[s], (uint32_t)((d >> 2) & 1));
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            uint32_t v[32], v1[32], v2[32];
            v2_ld32(lane_base + 96 + 96 * s, v);        // block kx = 0: this row's own
            v2_ld32(lane_base + 96 + 96 * s + 32, v1);  // block kx = 1: belongs to the row above (m - 1)
            v2_ld32(lane_base + 96 + 96 * s + 64, v2);  // block kx = 2: belongs to row m - 2
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) v2_arrive(&empty[s]);  // the slot is free as soon as it is in registers
            // out[m] = kx0[m] + kx1[m + 1] + kx2[m + 2]: shuffles inside the warp, the first two rows of the next warp
            // through shared memory (double-buffered by plane parity; one named barrier of the four epilogue warps)
            float (*xb)[3][32] = xch[grp][(d >> 1) & 1];
            if (lane < 2 && wq > 0) {
#pragma unroll
                for (int n = 0; n < 32; ++n) {
                    if (lane == 0) xb[wq][0][n] = __uint_as_float(v1[n]);
                    xb[wq][1 + lane][n] = __uint_as_float(v2[n]);
                }
            }
            if (grp == 0) asm volatile("bar.sync 1, 128;" ::: "memory");
            else asm volatile("bar.sync 2, 128;" ::: "memory");
            {
                // branch-free: every lane reads the (broadcast) hand-over values and selects -- a divergent branch per
                // element for the last two lanes cost more than the whole GEMM (measured: 0.69 of 1.2 ms)
                const int wn = wq < 3 ? wq + 1 : 3;  // the last warp's last rows (126, 127) are not outputs
                const uint32_t x1 = smem_u32(xb[wn][0]), x2 = smem_u32(xb[wn][lane == 31 ? 2 : 1]);
                const bool t1 = lane == 31, t2 = lane >= 30;
#pragma unroll
                for (int n = 0; n < 32; ++n) {
                    // raw shfl.sync: around __shfl_down_sync the compiler emitted a WARPSYNC + BSSY / BSYNC / BRA guard per
                    // element here (it cannot prove convergence behind the mbarrier spin loops): 6 x the instructions
                    uint32_t u1, u2;
                    asm volatile("shfl.sync.down.b32 %0, %1, 1, 0x1f, 0xffffffff;" : "=r"(u1) : "r"(v1[n]));
                    asm volatile("shfl.sync.down.b32 %0, %1, 2, 0x1f, 0xffffffff;" : "=r"(u2) : "r"(v2[n]));
                    // unconditional (volatile) loads + selects: a plain `t1 ? x1[n] : s1` became a branch around the load
                    // plus a WARPSYNC before the next shuffle, per element
                    float l1, l2;
                    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(l1) : "r"(x1 + 4 * n));
                    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(l2) : "r"(x2 + 4 * n));
                    const float a1 = t1 ? l1 : __uint_as_float(u1), a2 = t2 ? l2 : __uint_as_float(u2);
                    v[n] = __float_as_uint(__uint_as_float(v[n]) + a1 + a2);
                }
            }
            const int x = xt0 + m + d;
            const bool first = blockIdx.x == 0;
            // left-mask rows of the first tile: replace (xt = -2, -1) or correct (xt = 0, 1) the accumulator
            if (first && m < 4) {
                const float* cl = Cl + ((size_t)d * 4 + m) * 32;
#pragma unroll
                for (int n = 0; n < 32; ++n) v[n] = __float_as_uint(m < 2 ? cl[n] : __uint_as_float(v[n]) - cl[n]);
            }
            // first / last plane: the right-half term of the missing neighbour plane (kd = 0 / kd = 2) is not part of it
            if (d == 0 || d + 1 == Dq) {  // warp-uniform
                uint32_t t[32];
                if (d == 0) {
                    v2_ld32(lane_base + 0, t);
#pragma unroll
                    for (int n = 0; n < 32; ++n) v[n] = __float_as_uint(__uint_as_float(v[n]) - __uint_as_float(t[n]));
                }
                if (d + 1 == Dq) {
                    v2_ld32(lane_base + 64, t);
#pragma unroll
                    for (int n = 0; n < 32; ++n) v[n] = __float_as_uint(__uint_as_float(v[n]) - __uint_as_float(t[n]));
                }
            }
            T* o = out + ((size_t)b * kV2N * Dq + d) * HW + (size_t)y * W;
            if (m < kV2MT && x >= 0 && x < W) {
                const float* cr = Cr + (size_t)d * 32;
                const bool xr = x == W - 1;  // one row per plane
#pragma unroll
                for (int n = 0; n < 32; ++n) {
                    const float2 sc = ss[n];  // (scale, shift) or (1, 0): broadcast shared-memory read
                    const float c = cr[n];    // unconditional read + select (a branch per element costs more)
                    float val = __uint_as_float(v[n]) + qs[n] - (xr ? c : 0.f);
                    val = fmaf(val, sc.x, sc.y);
                    if (relu) val = fmaxf(val, 0.f);
                    st_from_f32(o + (size_t)n * cstride + x, val);
                }
            }
            // columns x <= d - 3 (shifted column <= -3): every tap is masked -> the epilogue of zero
            if (blockIdx.x == 0 && m <= d - 3 && m < W) {
#pragma unroll
                for (int n = 0; n < 32; ++n) {
                    float val = 0.f;
                    if (scale != nullptr) val = __ldg(shift + n);
                    if (relu) val = fmaxf(val, 0.f);
                    st_from_f32(o + (size_t)n * cstride + m, val);
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512));
}

template <typename T>
int volume_conv0_v2_launch(const T* L, const T* R, const float* wpacked, const float* scale, const float* shift,
                           T* out, int B, int H, int W, int Dq, int relu, cudaStream_t st, bool* done) {
    *done = false;
    if (Dq > kV2MaxDq || B > 65535 || H > 65535) return 0;
    cudaError_t e = cudaFuncSetAttribute(volume_conv0_v2_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, kV2Smem);
    if (e != cudaSuccess) return (int)e;
    // shifted columns -2 .. W - 1 (plane 0) must be covered
    dim3 grid((unsigned)ceil_div(W + 2, kV2MT), (unsigned)H, (unsigned)B);
    volume_conv0_v2_kernel<T><<<grid, kV2Threads, kV2Smem, st>>>(L, R, wpacked, scale, shift, out, B, H, W, Dq, relu);
    *done = true;
    return (int)cudaGetLastError();
}
template int volume_conv0_v2_launch<float>(const float*, const float*, const float*, const float*, const float*, float*, int,
                                           int, int, int, int, cudaStream_t, bool*);
template int volume_conv0_v2_launch<__nv_bfloat16>(const __nv_bfloat16*, const __nv_bfloat16*, const float*, const float*,
                                                   const float*, __nv_bfloat16*, int, int, int, int, int, cudaStream_t, bool*);
template int volume_conv0_v2_launch<__half>(const __half*, const __half*, const float*, const float*, const float*, __half*,
                                            int, int, int, int, int, cudaStream_t, bool*);

}  // namespace az
