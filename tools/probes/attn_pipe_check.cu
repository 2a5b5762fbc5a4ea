// Stand-alone check + timing of attention_pipe.cu against attention_tc.cu (the round-1 kernel) and a CPU
// double-precision reference on sampled (image, head) pairs.
// build (from tools/probes):
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo --expt-relaxed-constexpr \
//        attn_pipe_check.cu -o attn_pipe_check -L../../rajni_vit_b200/csrc -lrajni_b200 -lcuda -Xlinker -rpath='$ORIGIN/../../rajni_vit_b200/csrc'
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <vector>
#include "../../rajni_vit_b200/csrc/attention_pipe.cu"
namespace rajni {
int launch_attention_tc(const void* qkv, const int32_t* row_map, void* out, int B, int N_src, int Np,
                        int C, int H, float scale, int reverse, cudaStream_t stream);
}
extern "C" const char* rajni_last_error(void);

static float bf2f(__nv_bfloat16 v) { return __bfloat162float(v); }

struct Case { int B, N, Np, H; };

int main(int argc, char** argv) {
    std::vector<Case> cases = {{2, 17, 17, 2}, {3, 197, 197, 3}, {2, 197, 173, 12}, {2, 173, 152, 12}, {2, 152, 121, 12}, {2, 121, 87, 12},
                               {2, 64, 64, 1}, {2, 65, 65, 1}, {2, 197, 2, 3}, {3, 130, 129, 2}, {2, 192, 192, 2}, {2, 200, 193, 2},
                               {2, 224, 224, 2}, {2, 220, 209, 2}, {5, 128, 128, 3}, {4, 96, 96, 5}, {3, 150, 97, 4},
                               {256, 197, 197, 12}, {256, 197, 173, 12}, {256, 173, 152, 12}, {256, 152, 152, 12}, {256, 152, 121, 12},
                               {256, 121, 87, 12}, {256, 87, 87, 12}, {32, 197, 197, 12}, {64, 197, 197, 6}};
    if (argc >= 5) { cases.clear(); cases.push_back({atoi(argv[1]), atoi(argv[2]), atoi(argv[3]), atoi(argv[4])}); }
    int bad = 0;
    for (const Case& c : cases) {
        const int B = c.B, N = c.N, Np = c.Np, H = c.H, C = H * 64;
        std::vector<__nv_bfloat16> h((size_t)B * N * 3 * C);
        srand(B * 131 + N * 7 + Np);
        for (auto& x : h) x = __float2bfloat16((rand() % 4001 - 2000) / 700.f);
        std::vector<int> rm((size_t)B * Np);
        for (int b = 0; b < B; ++b) for (int j = 0; j < Np; ++j) rm[b * Np + j] = b * N + (j == 0 ? 0 : 1 + ((j - 1) * (N - 1)) / (Np - 1 > 0 ? Np - 1 : 1));
        __nv_bfloat16 *qkv, *out0, *out1; int* rmap;
        cudaMalloc(&qkv, h.size() * 2); cudaMalloc(&out0, (size_t)B * Np * C * 2); cudaMalloc(&out1, (size_t)B * Np * C * 2); cudaMalloc(&rmap, rm.size() * 4);
        cudaMemcpy(qkv, h.data(), h.size() * 2, cudaMemcpyHostToDevice);
        cudaMemcpy(rmap, rm.data(), rm.size() * 4, cudaMemcpyHostToDevice);
        cudaMemset(out0, 0xff, (size_t)B * Np * C * 2); cudaMemset(out1, 0xff, (size_t)B * Np * C * 2);
        const int32_t* rmp = Np < N ? rmap : nullptr;
        int rc0 = rajni::launch_attention_tc(qkv, rmp, out0, B, N, Np, C, H, 0.125f, 0, 0);
        cudaError_t e0 = cudaDeviceSynchronize();
        int rc1 = rajni::launch_attention_pipe(qkv, rmp, out1, B, N, Np, C, H, 0.125f, 0, 0);
        cudaError_t e1 = cudaDeviceSynchronize();
        if (rc0 < 0 || rc1 < 0 || e0 != cudaSuccess || e1 != cudaSuccess) {
            printf("B=%d N=%d Np=%d H=%d: rc %d %d cuda %s / %s (%s)\n", B, N, Np, H, rc0, rc1, cudaGetErrorString(e0), cudaGetErrorString(e1), rajni_last_error());
            return 2;
        }
        std::vector<__nv_bfloat16> o0((size_t)B * Np * C), o1(o0.size());
        cudaMemcpy(o0.data(), out0, o0.size() * 2, cudaMemcpyDeviceToHost);
        cudaMemcpy(o1.data(), out1, o1.size() * 2, cudaMemcpyDeviceToHost);
        double dmax = 0; size_t nbad = 0;
        for (size_t i = 0; i < o0.size(); ++i) {
            const float a = bf2f(o0[i]), b = bf2f(o1[i]);
            const double d = fabs((double)a - b);
            // (two kernels, each within the tolerance of the exact result: twice that between them)
            if (!(d <= 2 * (0.0157 * fabs(a) + 4e-3))) { if (nbad < 4) printf("  bad at row %zu col %zu: tc %.5f pipe %.5f\n", i / C, i % C, a, b); ++nbad; }
            if (d > dmax || d != d) dmax = d;
        }
        // CPU double reference on a few (image, head) pairs, both directions of traversal covered by rc1 above
        double cmax = 0;
        for (int s = 0; s < 3; ++s) {
            const int b = (s * 7919) % B, hh = (s * 31 + 1) % H;
            std::vector<double> pr(Np);
            for (int i = 0; i < Np; i += (Np > 40 ? 13 : 1)) {
                const size_t qi = (size_t)(Np < N ? rm[b * Np + i] : b * N + i) * 3 * C + hh * 64;
                double mx = -1e300;
                for (int j = 0; j < Np; ++j) {
                    const size_t kj = (size_t)(Np < N ? rm[b * Np + j] : b * N + j) * 3 * C + C + hh * 64;
                    double sdot = 0;
                    for (int d = 0; d < 64; ++d) sdot += (double)bf2f(h[qi + d]) * bf2f(h[kj + d]);
                    pr[j] = sdot * 0.125;
                    mx = fmax(mx, pr[j]);
                }
                double sum = 0;
                for (int j = 0; j < Np; ++j) { pr[j] = exp(pr[j] - mx); sum += pr[j]; }
                for (int d = 0; d < 64; ++d) {
                    double o = 0;
                    for (int j = 0; j < Np; ++j) {
                        const size_t vj = (size_t)(Np < N ? rm[b * Np + j] : b * N + j) * 3 * C + 2 * C + hh * 64;
                        o += pr[j] * bf2f(h[vj + d]);
                    }
                    o /= sum;
                    const double got = bf2f(o1[((size_t)b * Np + i) * C + hh * 64 + d]);
                    const double err = fabs(got - o) / (fabs(o) * 0.0157 + 4e-3);
                    if (err > cmax || err != err) cmax = err;
                }
            }
        }
        // timing
        float ms0 = 0, ms1 = 0;
        if (B >= 32) {
            cudaEvent_t a, b2; cudaEventCreate(&a); cudaEventCreate(&b2);
            const int it = 20;
            for (int k = 0; k < 3; ++k) rajni::launch_attention_tc(qkv, rmp, out0, B, N, Np, C, H, 0.125f, 0, 0);
            cudaEventRecord(a);
            for (int k = 0; k < it; ++k) rajni::launch_attention_tc(qkv, rmp, out0, B, N, Np, C, H, 0.125f, 0, 0);
            cudaEventRecord(b2); cudaEventSynchronize(b2); cudaEventElapsedTime(&ms0, a, b2); ms0 /= it;
            for (int k = 0; k < 3; ++k) rajni::launch_attention_pipe(qkv, rmp, out1, B, N, Np, C, H, 0.125f, 0, 0);
            cudaEventRecord(a);
            for (int k = 0; k < it; ++k) rajni::launch_attention_pipe(qkv, rmp, out1, B, N, Np, C, H, 0.125f, 0, 0);
            cudaEventRecord(b2); cudaEventSynchronize(b2); cudaEventElapsedTime(&ms1, a, b2); ms1 /= it;
        }
        const bool ok = cmax <= 1.0;            /* (vs tc is informative: both round P to bf16 independently) */
        bad += !ok;
        printf("B=%3d N=%3d Np=%3d H=%2d: vs tc max|d|=%.4f bad=%zu  cpu err/tol=%.3f  %s", B, N, Np, H, dmax, nbad, cmax, ok ? "ok" : "FAIL");
        if (B >= 32) printf("   tc %.1f us  pipe %.1f us  (%.2fx, %.0f TF/s)", ms0 * 1e3, ms1 * 1e3, ms0 / ms1, 4.0 * B * Np * Np * C / (ms1 * 1e-3) / 1e12);
        printf("\n");
        fflush(stdout);
        cudaFree(qkv); cudaFree(out0); cudaFree(out1); cudaFree(rmap);
    }
    // NaN isolation (dense call): image 1 all-NaN must not touch image 0's output
    {
        const int B = 2, N = 197, H = 2, C = 128;
        std::vector<__nv_bfloat16> h((size_t)B * N * 3 * C);
        for (size_t i = 0; i < h.size(); ++i) h[i] = i < h.size() / 2 ? __float2bfloat16(((int)(i % 97) - 48) / 40.f) : __float2bfloat16(NAN);
        __nv_bfloat16 *qkv, *out; cudaMalloc(&qkv, h.size() * 2); cudaMalloc(&out, (size_t)B * N * C * 2);
        cudaMemcpy(qkv, h.data(), h.size() * 2, cudaMemcpyHostToDevice);
        rajni::launch_attention_pipe(qkv, nullptr, out, B, N, N, C, H, 0.125f, 0, 0);
        cudaDeviceSynchronize();
        std::vector<__nv_bfloat16> o((size_t)N * C);
        cudaMemcpy(o.data(), out, o.size() * 2, cudaMemcpyDeviceToHost);
        int nan0 = 0;
        for (auto v : o) nan0 += bf2f(v) != bf2f(v);
        printf("NaN isolation: %d NaN values in image 0's output (%s)\n", nan0, nan0 ? "FAIL" : "ok");
        bad += nan0 != 0;
    }
    printf(bad ? "FAILED (%d)\n" : "all ok\n", bad);
    return bad ? 1 : 0;
}
