// probe_gemm.cu -- stand-alone check of k_dense (rd_gemm.cuh) against a float64 CPU product, run on the GPU box:
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -o gpurun_out/probe_gemm tools/probe_gemm.cu
//   timeout 120 gpurun_out/probe_gemm
// Exercises the three plumbing shapes the Dreamer policy uses: one phase / one slab (Dense), two phases over two A
// sources (concat input), three slabs into four accumulators (GRU).  Prints max |error| relative to the row scale.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "../racing_dreamer_b200/csrc/rd_gemm.cuh"

#define CK(x)                                                                                   \
  do {                                                                                          \
    cudaError_t e_ = (x);                                                                       \
    if (e_ != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); exit(2); } \
  } while (0)

static float frand() { return (float)rand() / (float)RAND_MAX * 2.f - 1.f; }
static double elu(double x) { return x > 0 ? x : std::expm1(x); }

int main() {
  srand(1);
  int fails = 0;
  // ---------------- T1: dense ELU, M = 300 (partial tile), K = 232, N = 400 ----------------
  {
    const int M = 300, K = 232, N = 400;
    std::vector<float> A((size_t)M * K), W((size_t)N * K), b(N);
    for (auto& x : A) x = frand();
    for (auto& x : W) x = frand() * 0.1f;
    for (auto& x : b) x = frand() * 0.1f;
    float *dA, *dW, *db, *dO;
    CK(cudaMalloc(&dA, A.size() * 4)); CK(cudaMalloc(&dW, W.size() * 4)); CK(cudaMalloc(&db, N * 4)); CK(cudaMalloc(&dO, (size_t)M * N * 4));
    CK(cudaMemcpy(dA, A.data(), A.size() * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dW, W.data(), W.size() * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(db, b.data(), N * 4, cudaMemcpyHostToDevice));
    CK(cudaMemset(dO, 0, (size_t)M * N * 4));
    CUtensorMap ma, mw, mo;
    if (!gm_make_map(&ma, dA, K, M, K, GM_BM) || !gm_make_map(&mw, dW, K, N, K, GM_BN) || !gm_make_map(&mo, dO, N, M, N, GM_BM)) {
      printf("T1 map encode failed\n"); return 3;
    }
    GemmArgs g{};
    g.M = M; g.N = N; g.n_phases = 1; g.n_acc = 1;
    g.ph[0].k_blocks = (K + 31) / 32; g.ph[0].nb = 1; g.ph[0].w_row0[0] = 0; g.ph[0].acc[0] = 0;
    g.bias = db; g.out = dO; g.ldo = N; g.act = 1;
    GemmMaps maps{};
    maps.a[0] = ma; maps.w[0] = mw; maps.o[0] = mo;
    CK((gm_launch<EPI_DENSE, 1, 4, 4>(maps, g, 0)));
    CK(cudaDeviceSynchronize());
    std::vector<float> O((size_t)M * N);
    CK(cudaMemcpy(O.data(), dO, O.size() * 4, cudaMemcpyDeviceToHost));
    double worst = 0;
    for (int i = 0; i < M; ++i)
      for (int j = 0; j < N; ++j) {
        double s = b[j], sc = 0;
        for (int k = 0; k < K; ++k) { s += (double)A[(size_t)i * K + k] * W[(size_t)j * K + k]; sc += std::fabs((double)A[(size_t)i * K + k] * W[(size_t)j * K + k]); }
        double err = std::fabs(elu(s) - O[(size_t)i * N + j]) / (sc + 1e-6);
        if (err > worst) worst = err;
      }
    printf("T1 dense   M=%d K=%d N=%d  max err / sum|a w| = %.3e  %s\n", M, K, N, worst, worst < 2e-3 ? "ok" : "FAIL");
    fails += !(worst < 2e-3);
  }
  // ---------------- T2: two phases: [A0 (200 of ld 232, offset 32) | A1 (1080)] @ W[200][1280], linear ----------------
  {
    const int M = 200, K0 = 200, K1 = 1080, N = 200, LD0 = 232;
    std::vector<float> F((size_t)M * LD0), L((size_t)M * K1), W((size_t)N * (K0 + K1)), b(N);
    for (auto& x : F) x = frand();
    for (auto& x : L) x = frand() * 7.f + 7.5f;
    for (auto& x : W) x = frand() * 0.05f;
    for (auto& x : b) x = frand();
    float *dF, *dL, *dW, *db, *dO;
    CK(cudaMalloc(&dF, F.size() * 4)); CK(cudaMalloc(&dL, L.size() * 4)); CK(cudaMalloc(&dW, W.size() * 4)); CK(cudaMalloc(&db, N * 4));
    CK(cudaMalloc(&dO, (size_t)M * N * 4));
    CK(cudaMemcpy(dF, F.data(), F.size() * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dL, L.data(), L.size() * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dW, W.data(), W.size() * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(db, b.data(), N * 4, cudaMemcpyHostToDevice));
    CUtensorMap ma0, ma1, mw, mo;
    if (!gm_make_map(&ma0, dF + 32, K0, M, LD0, GM_BM) || !gm_make_map(&ma1, dL, K1, M, K1, GM_BM) ||
        !gm_make_map(&mw, dW, K0 + K1, N, K0 + K1, GM_BN) || !gm_make_map(&mo, dO, N, M, N, GM_BM)) { printf("T2 map encode failed\n"); return 3; }
    GemmArgs g{};
    g.M = M; g.N = N; g.n_phases = 2; g.n_acc = 1;
    g.ph[0].k_blocks = (K0 + 31) / 32; g.ph[0].nb = 1; g.ph[0].w_k0 = 0;
    g.ph[1].k_blocks = (K1 + 31) / 32; g.ph[1].nb = 1; g.ph[1].w_k0 = K0; g.ph[1].a_map = 1;
    g.bias = db; g.out = dO; g.ldo = N; g.act = 0;
    GemmMaps maps{};
    maps.a[0] = ma0; maps.a[1] = ma1; maps.w[0] = mw; maps.o[0] = mo;
    CK((gm_launch<EPI_DENSE, 1, 4, 4>(maps, g, 0)));
    CK(cudaDeviceSynchronize());
    std::vector<float> O((size_t)M * N);
    CK(cudaMemcpy(O.data(), dO, O.size() * 4, cudaMemcpyDeviceToHost));
    double worst = 0;
    for (int i = 0; i < M; ++i)
      for (int j = 0; j < N; ++j) {
        double s = b[j], sc = 0;
        for (int k = 0; k < K0; ++k) { double t = (double)F[(size_t)i * LD0 + 32 + k] * W[(size_t)j * (K0 + K1) + k]; s += t; sc += std::fabs(t); }
        for (int k = 0; k < K1; ++k) { double t = (double)L[(size_t)i * K1 + k] * W[(size_t)j * (K0 + K1) + K0 + k]; s += t; sc += std::fabs(t); }
        double err = std::fabs(s - O[(size_t)i * N + j]) / (sc + 1e-6);
        if (err > worst) worst = err;
      }
    printf("T2 concat  M=%d K=%d+%d N=%d  max err / sum|a w| = %.3e  %s\n", M, K0, K1, N, worst, worst < 2e-3 ? "ok" : "FAIL");
    fails += !(worst < 2e-3);
  }
  // ---------------- T3: GRU cell, H = 200 ----------------
  {
    const int M = 333, H = 200, LD = 232;
    std::vector<float> X((size_t)M * H), F((size_t)M * LD), Wk((size_t)3 * H * H), Wr((size_t)3 * H * H), b(6 * H);
    for (auto& x : X) x = frand();
    for (auto& x : F) x = frand();
    for (auto& x : Wk) x = frand() * 0.1f;
    for (auto& x : Wr) x = frand() * 0.1f;
    for (auto& x : b) x = frand() * 0.2f;
    float *dX, *dF, *dWk, *dWr, *db, *dO;
    CK(cudaMalloc(&dX, X.size() * 4)); CK(cudaMalloc(&dF, F.size() * 4)); CK(cudaMalloc(&dWk, Wk.size() * 4)); CK(cudaMalloc(&dWr, Wr.size() * 4));
    CK(cudaMalloc(&db, b.size() * 4)); CK(cudaMalloc(&dO, (size_t)M * LD * 4));
    CK(cudaMemcpy(dX, X.data(), X.size() * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dF, F.data(), F.size() * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dWk, Wk.data(), Wk.size() * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dWr, Wr.data(), Wr.size() * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(db, b.data(), b.size() * 4, cudaMemcpyHostToDevice));
    CK(cudaMemset(dO, 0, (size_t)M * LD * 4));
    CUtensorMap mx, mh, mwk, mwr, mo;
    if (!gm_make_map(&mx, dX, H, M, H, GM_BM) || !gm_make_map(&mh, dF + 32, H, M, LD, GM_BM) ||
        !gm_make_map(&mwk, dWk, H, 3 * H, H, GM_BN) || !gm_make_map(&mwr, dWr, H, 3 * H, H, GM_BN) ||
        !gm_make_map(&mo, dO + 32, H, M, LD, GM_BM)) { printf("T3 map encode failed\n"); return 3; }
    GemmArgs g{};
    g.M = M; g.N = H; g.n_phases = 2; g.n_acc = 1;
    for (int p = 0; p < 2; ++p) {
      g.ph[p].k_blocks = (H + 31) / 32; g.ph[p].nb = 3; g.ph[p].a_map = p; g.ph[p].w_map = p;
      g.ph[p].w_row0[0] = 0; g.ph[p].w_row0[1] = H; g.ph[p].w_row0[2] = 2 * H;
      g.ph[p].acc[0] = 0; g.ph[p].acc[1] = 1; g.ph[p].acc[2] = p == 0 ? 2 : 3;
    }
    g.bias = db; g.out = dO + 32; g.ldo = LD; g.hold = dF + 32; g.ldh = LD;
    GemmMaps maps{};
    maps.a[0] = mx; maps.a[1] = mh; maps.w[0] = mwk; maps.w[1] = mwr; maps.o[0] = mo;
    CK((gm_launch<EPI_GRU, 3, 8, 4>(maps, g, 0)));
    CK(cudaDeviceSynchronize());
    std::vector<float> O((size_t)M * LD);
    CK(cudaMemcpy(O.data(), dO, O.size() * 4, cudaMemcpyDeviceToHost));
    double worst = 0;
    for (int i = 0; i < M; ++i)
      for (int c = 0; c < H; ++c) {
        double gx[3], gh[3];
        for (int q = 0; q < 3; ++q) {
          double sx = b[q * H + c], sh = b[3 * H + q * H + c];
          for (int k = 0; k < H; ++k) {
            sx += (double)X[(size_t)i * H + k] * Wk[(size_t)(q * H + c) * H + k];
            sh += (double)F[(size_t)i * LD + 32 + k] * Wr[(size_t)(q * H + c) * H + k];
          }
          gx[q] = sx; gh[q] = sh;
        }
        double z = 1 / (1 + std::exp(-(gx[0] + gh[0]))), r = 1 / (1 + std::exp(-(gx[1] + gh[1])));
        double hh = std::tanh(gx[2] + r * gh[2]);
        double h = z * F[(size_t)i * LD + 32 + c] + (1 - z) * hh;
        double err = std::fabs(h - O[(size_t)i * LD + 32 + c]);
        if (err > worst) worst = err;
      }
    printf("T3 gru     M=%d H=%d  max |err| = %.3e  %s\n", M, H, worst, worst < 5e-3 ? "ok" : "FAIL");
    fails += !(worst < 5e-3);
  }
  printf(fails ? "PROBE FAILED (%d)\n" : "PROBE OK\n", fails);
  return fails ? 1 : 0;
}
