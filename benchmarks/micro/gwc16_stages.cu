// Stage count of the 16-bit systolic gwc backward (activezero_b200/csrc/gwc_volume.cu, not part of the library build;
// DESIGN.md §4.15).  The kernel is bound by the bytes its stage rings keep in flight, and a 16-bit stage holds half the
// bytes of an fp32 one: this times gwc_bwd_systolic_kernel<bf16, 4, 128, S, false> for S = 5, 6, 8, 10 against the fp32
// kernel the library runs (S = 5) at config 2 (B = 8, C = 32, G = 8, 136x240, Dq = 48; gvol 200 MB in bf16, past L2),
// after checking that every S writes the same gradients.  Arms alternated: 10 windows of 20 launches after one warm-up
// window; one JSON line per arm with the median and the fraction of a device-to-device copy measured in the same run.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -o gwc16_stages gwc16_stages.cu && ./gwc16_stages
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <vector>

#include "../../activezero_b200/csrc/gwc_volume.cu"

constexpr int kB = 8, kC = 32, kG = 8, kH = 136, kW = 240, kDq = 48, kCPG = kC / kG;

template <typename T, int S>
static void launch(const void* g, const void* L, const void* R, void* gL, void* gR) {
    constexpr int NT = 128;
    const int rows = NT / (kW / 4);
    const size_t smem = (size_t)(S * 4 + kCPG) * NT * sizeof(GwcQuad<T>);
    auto kern = gwc_bwd_systolic_kernel<T, kCPG, NT, S, false>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    dim3 grid((unsigned)ceil_div(kH, rows), kG, kB);
    kern<<<grid, NT, smem>>>((const T*)g, (const T*)L, (const T*)R, (T*)gL, (T*)gR, kC, kG, kH, kW, kDq, rows);
}

int main() {
    const size_t nf = (size_t)kB * kC * kH * kW, ng = (size_t)kB * kG * kDq * kH * kW;
    std::vector<float> hf(2 * nf), hg(ng);
    uint32_t s = 12345u;
    auto rnd = [&]() { s = s * 1664525u + 1013904223u; return (float)((s >> 8) & 0xffff) / 32768.f - 1.f; };
    for (auto& v : hf) v = rnd();
    for (auto& v : hg) v = rnd();
    std::vector<__nv_bfloat16> hf16(2 * nf), hg16(ng);
    for (size_t i = 0; i < 2 * nf; ++i) hf16[i] = __float2bfloat16_rn(hf[i]);
    for (size_t i = 0; i < ng; ++i) hg16[i] = __float2bfloat16_rn(hg[i]);
    void *f32, *g32, *o32, *f16, *g16, *o16, *ref16, *cpy;
    cudaMalloc(&f32, 2 * nf * 4); cudaMalloc(&g32, ng * 4); cudaMalloc(&o32, 2 * nf * 4);
    cudaMalloc(&f16, 2 * nf * 2); cudaMalloc(&g16, ng * 2); cudaMalloc(&o16, 2 * nf * 2); cudaMalloc(&ref16, 2 * nf * 2);
    const size_t cpy_bytes = (size_t)1 << 30;
    cudaMalloc(&cpy, 2 * cpy_bytes);
    cudaMemcpy(f32, hf.data(), 2 * nf * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(g32, hg.data(), ng * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(f16, hf16.data(), 2 * nf * 2, cudaMemcpyHostToDevice);
    cudaMemcpy(g16, hg16.data(), ng * 2, cudaMemcpyHostToDevice);
    cudaMemset(cpy, 0, 2 * cpy_bytes);
    using BF = __nv_bfloat16;
    char* F16 = (char*)f16; char* O16 = (char*)o16; char* F32 = (char*)f32; char* O32 = (char*)o32;
    const int nS = 4;
    const char* names[nS + 2] = {"bf16_S5", "bf16_S6", "bf16_S8", "bf16_S10", "fp32_S5", "d2d_copy_1GiB"};
    auto run = [&](int a) {
        switch (a) {
            case 0: launch<BF, 5>(g16, F16, F16 + nf * 2, O16, O16 + nf * 2); break;
            case 1: launch<BF, 6>(g16, F16, F16 + nf * 2, O16, O16 + nf * 2); break;
            case 2: launch<BF, 8>(g16, F16, F16 + nf * 2, O16, O16 + nf * 2); break;
            case 3: launch<BF, 10>(g16, F16, F16 + nf * 2, O16, O16 + nf * 2); break;
            case 4: launch<float, 5>(g32, F32, F32 + nf * 4, O32, O32 + nf * 4); break;
            default: cudaMemcpyAsync((char*)cpy + cpy_bytes, cpy, cpy_bytes, cudaMemcpyDeviceToDevice); break;
        }
    };
    // every stage count writes the same gradients
    run(0);
    cudaMemcpy(ref16, o16, 2 * nf * 2, cudaMemcpyDeviceToDevice);
    std::vector<unsigned short> a(2 * nf), b(2 * nf);
    cudaMemcpy(a.data(), ref16, 2 * nf * 2, cudaMemcpyDeviceToHost);
    for (int k = 1; k < nS; ++k) {
        cudaMemset(o16, 0xff, 2 * nf * 2);
        run(k);
        cudaMemcpy(b.data(), o16, 2 * nf * 2, cudaMemcpyDeviceToHost);
        size_t diff = 0;
        for (size_t i = 0; i < 2 * nf; ++i) diff += a[i] != b[i];
        printf("{\"check\": \"%s vs bf16_S5\", \"elements_differing\": %zu}\n", names[k], diff);
    }
    cudaError_t err = cudaDeviceSynchronize();
    if (err != cudaSuccess) { printf("{\"error\": \"%s\"}\n", cudaGetErrorString(err)); return 1; }
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    const int nA = nS + 2, windows = 10, per = 20;
    std::vector<std::vector<float>> ms(nA);
    for (int w = 0; w <= windows; ++w) {
        for (int k = 0; k < nA; ++k) {
            cudaEventRecord(e0);
            for (int i = 0; i < per; ++i) run(k);
            cudaEventRecord(e1);
            cudaEventSynchronize(e1);
            float t = 0.f;
            cudaEventElapsedTime(&t, e0, e1);
            if (w > 0) ms[k].push_back(t / per);
        }
    }
    auto med = [](std::vector<float> v) { std::sort(v.begin(), v.end()); return v[v.size() / 2]; };
    const double copy_Bps = 2.0 * cpy_bytes / (med(ms[nA - 1]) * 1e-3);
    // algorithmic bytes of the backward: s * (G*Dq*HW + 4*C*HW) * B
    const double hw = (double)kH * kW;
    const double bytes16 = 2.0 * kB * (kG * kDq * hw + 4.0 * kC * hw), bytes32 = 2.0 * bytes16;
    for (int k = 0; k < nA; ++k) {
        const double m = med(ms[k]);
        const double bytes = k < nS ? bytes16 : (k == nS ? bytes32 : 2.0 * cpy_bytes);
        printf("{\"arm\": \"%s\", \"median_ms\": %.4f, \"min_ms\": %.4f, \"max_ms\": %.4f, \"GBps\": %.0f, "
               "\"fraction_of_copy_peak\": %.3f}\n",
               names[k], m, *std::min_element(ms[k].begin(), ms[k].end()), *std::max_element(ms[k].begin(), ms[k].end()),
               bytes / (m * 1e-3) / 1e9, bytes / (m * 1e-3) / copy_Bps);
    }
    return 0;
}
