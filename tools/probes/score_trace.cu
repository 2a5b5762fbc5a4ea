// Event timeline (globaltimer, ns) of one CTA of the overlapped score kernel: per unit wait/compute, and the phases of each tail.
// build: nvcc -O3 -std=c++17 --expt-relaxed-constexpr -gencode arch=compute_100a,code=sm_100a -DRAJNI_SCORE_TRACE -I../../rajni_vit_b200/csrc score_trace.cu -o score_trace
#include <cstdio>
#include <cstdlib>
#include <vector>
#include "../../rajni_vit_b200/csrc/score_select.cu"
namespace rajni { void set_error(const char*, ...) {} void count_launch(int) {} int check_launch(const char*) { return cudaGetLastError() == cudaSuccess ? 0 : -2; }
                  bool pdl_enabled() { return false; } int current_device() { return 0; } }
int main(int argc, char** argv) {
    const int B = argc > 1 ? atoi(argv[1]) : 256, N = argc > 2 ? atoi(argv[2]) : 197, H = argc > 3 ? atoi(argv[3]) : 12, C = H * 64;
    const int cta = argc > 4 ? atoi(argv[4]) : 0;
    const int keep = (int)(0.88 * (N - 1));
    std::vector<__nv_bfloat16> h((size_t)B * N * 3 * C);
    srand(1);
    for (auto& x : h) x = __float2bfloat16((rand() % 2001 - 1000) / 500.f);
    __nv_bfloat16* qkv[3]; int* idx; float* nxt; int* rmap; void* ws;
    for (auto& q : qkv) { cudaMalloc(&q, h.size() * 2); cudaMemcpy(q, h.data(), h.size() * 2, cudaMemcpyHostToDevice); }
    cudaMalloc(&idx, (size_t)B * (keep + 1) * 4); cudaMalloc(&nxt, (size_t)B * (keep + 1) * 4); cudaMalloc(&rmap, (size_t)B * (keep + 1) * 4);
    size_t wb = rajni_score_select_workspace_bytes(B, N, C, H);
    cudaMalloc(&ws, wb); cudaMemset(ws, 0, wb);
    cudaMemcpyToSymbol(rajni::g_sc_trace_cta, &cta, sizeof(int));
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    for (int i = 0; i < 6; ++i) {
        if (i == 5) cudaEventRecord(e0);
        int rc = rajni_score_select_prefix(qkv[i % 3], B, N, C, H, 1, keep, 1e-6f, nullptr, idx, nxt, rmap, ws, wb, 0);
        if (rc) { printf("rc=%d\n", rc); return 1; }
    }
    cudaEventRecord(e1);
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { printf("error: %s\n", cudaGetErrorString(e)); return 1; }
    float ms; cudaEventElapsedTime(&ms, e0, e1);
    printf("B=%d N=%d H=%d: last launch %.1f us; CTA %d timeline (ns from its first stamp)\n", B, N, H, ms * 1e3, cta);
    static long long tr[64 * 16];
    cudaMemcpyFromSymbol(tr, rajni::g_sc_trace, sizeof(tr));
    const char* names[11] = {"unit:beg", "unit:done", "tail:go", "tail:copied", "t:mu", "t:r", "t:softmax", "t:zstat", "t:score", "t:select", "t:end"};
    printf("unit");
    for (auto n : names) printf(" %11s", n);
    printf("\n");
    const long long t0 = tr[0];
    for (int u = 0; u < 64; ++u) {          // rows 0..31: units; rows 32..: the tails this CTA ran
        bool any = false;
        for (int s = 0; s < 11; ++s) any |= tr[u * 16 + s] != 0;
        if (!any) continue;
        printf("%4d", u);
        for (int s = 0; s < 11; ++s) printf(" %11lld", tr[u * 16 + s] >= t0 && tr[u * 16 + s] ? tr[u * 16 + s] - t0 : -1);
        printf("\n");
    }
    return 0;
}
