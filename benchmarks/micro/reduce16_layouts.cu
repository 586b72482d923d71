// The reduce kernel of the volume-free backward (activezero_b200/csrc/volume_conv_bwd.cu, not part of the library
// build) in its three forms on the same g at the two shapes of benchmarks/volume_conv_train.py: fp32 one column per
// thread, 16-bit one column per thread, 16-bit two columns per thread (DESIGN.md §4.13).  Checks that the two 16-bit
// forms write identical planes, then times them alternated: 10 windows of 50 launches after one warm-up window.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -o reduce16_layouts reduce16_layouts.cu && ./reduce16_layouts
#include <cstdio>
#include <vector>
#include <algorithm>
#include <cstring>
#include "../../activezero_b200/csrc/volume_conv_bwd.cu"

template <typename T, bool TWO>
static void launch(const void* g, float* planes, int B, int H, int W, int Dq) {
    if constexpr (TWO) {
        dim3 grid((unsigned)(B * kVbC * H), (unsigned)ceil_div(W, 2 * kVbRedT));
        vcb_reduce2_kernel<T><<<grid, kVbRedT>>>((const T*)g, planes, B, H, W, Dq);
    } else {
        dim3 grid((unsigned)(B * kVbC * H), (unsigned)ceil_div(W, kVbRedT));
        vcb_reduce_kernel<T><<<grid, kVbRedT>>>((const T*)g, planes, B, H, W, Dq);
    }
}

int main() {
    const int shapes[2][4] = {{2, 64, 128, 48}, {2, 136, 240, 48}};
    for (auto& s : shapes) {
        const int B = s[0], H = s[1], W = s[2], Dq = s[3];
        const size_t n = (size_t)B * 32 * Dq * H * W, np = (size_t)18 * B * 32 * H * W;
        void *g32, *g16; float *p1, *p2;
        cudaMalloc(&g32, n * 4); cudaMalloc(&g16, n * 2); cudaMalloc(&p1, np * 4); cudaMalloc(&p2, np * 4);
        std::vector<unsigned short> h(n);
        uint32_t st = 12345u;
        for (size_t i = 0; i < n; ++i) { st = st * 1664525u + 1013904223u; h[i] = (unsigned short)(0x3c00 | ((st >> 9) & 0x3ff) | ((st >> 31) << 15)); }
        cudaMemcpy(g16, h.data(), n * 2, cudaMemcpyHostToDevice);
        cudaMemset(g32, 0, n * 4);
        // check: both 16-bit forms give identical planes
        for (int dt = 0; dt < 2; ++dt) {
            if (dt == 0) { launch<__nv_bfloat16, false>(g16, p1, B, H, W, Dq); launch<__nv_bfloat16, true>(g16, p2, B, H, W, Dq); }
            else { launch<__half, false>(g16, p1, B, H, W, Dq); launch<__half, true>(g16, p2, B, H, W, Dq); }
            cudaDeviceSynchronize();
            std::vector<float> a(np), b(np);
            cudaMemcpy(a.data(), p1, np * 4, cudaMemcpyDeviceToHost);
            cudaMemcpy(b.data(), p2, np * 4, cudaMemcpyDeviceToHost);
            size_t bad = 0;
            for (size_t i = 0; i < np; ++i) bad += memcmp(&a[i], &b[i], 4) != 0;
            printf("{\"shape\": \"B%d_%dx%d_Dq%d\", \"dtype\": \"%s\", \"planes_differing\": %zu}\n", B, H, W, Dq, dt ? "fp16" : "bf16", bad);
        }
        const char* names[5] = {"fp32_1col", "bf16_1col", "bf16_2col", "fp16_1col", "fp16_2col"};
        std::vector<float> t[5];
        cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
        const int iters = 50;
        for (int rep = 0; rep < 11; ++rep) {
            for (int k = 0; k < 5; ++k) {
                cudaEventRecord(e0);
                for (int it = 0; it < iters; ++it) {
                    switch (k) {
                        case 0: launch<float, false>(g32, p1, B, H, W, Dq); break;
                        case 1: launch<__nv_bfloat16, false>(g16, p1, B, H, W, Dq); break;
                        case 2: launch<__nv_bfloat16, true>(g16, p1, B, H, W, Dq); break;
                        case 3: launch<__half, false>(g16, p1, B, H, W, Dq); break;
                        case 4: launch<__half, true>(g16, p1, B, H, W, Dq); break;
                    }
                }
                cudaEventRecord(e1); cudaEventSynchronize(e1);
                float ms; cudaEventElapsedTime(&ms, e0, e1);
                if (rep > 0) t[k].push_back(ms / iters);
            }
        }
        for (int k = 0; k < 5; ++k) {
            std::sort(t[k].begin(), t[k].end());
            const double bytes = (double)n * (k == 0 ? 4 : 2) + (double)np * 4;
            const double med = t[k][t[k].size() / 2];
            printf("{\"shape\": \"B%d_%dx%d_Dq%d\", \"kernel\": \"%s\", \"median_ms\": %.4f, \"min_ms\": %.4f, \"GBps_on_g_in_planes_out\": %.0f}\n",
                   B, H, W, Dq, names[k], med, t[k][0], bytes / med / 1e6);
        }
        printf("{\"error\": \"%s\"}\n", cudaGetErrorString(cudaGetLastError()));
        cudaFree(g32); cudaFree(g16); cudaFree(p1); cudaFree(p2);
    }
    return 0;
}
