// Stand-alone timing harness for k_relax_ws<4,4,WPC,false> (the production relax kernel) on a synthetic
// n x n x 4 level: builds in seconds (one instantiation), prints the per-step time of worker 0, the
// lag between neighbouring workers and a checksum of the result (must not change between variants).
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -fmad=false -o relax_bench relax_bench.cu
//   ./relax_bench [n=4096] [nsweeps=4] [repetitions=0]
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include <algorithm>
#include "../../msom_b200/csrc/mg_kernels.cuh"
#ifndef BWPC
#define BWPC 4
#endif
#define CKC(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e), __FILE__, __LINE__); exit(1); } } while (0)
__global__ void k_fill(unsigned long long *p, size_t n, unsigned long long v) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = v;
}
int main(int argc, char **argv) {
  const int n = argc > 1 ? atoi(argv[1]) : 4096, nsw = argc > 2 ? atoi(argv[2]) : 4;
  constexpr int NL = 4, K = 4;
  using Cfg = WsCfg<NL, K>;
  Geom g{};
  g.nx = g.ny = n; g.bc = 0; g.pitch = msqg_pitch(n); g.plane = (size_t)(n + 2) * g.pitch; g.Delta = 80.0 / n; g.rD = 1. / g.Delta;
  RelaxCoef<NL> C;
  {
    const double Delta = g.Delta, dh[4] = {0.05, 0.1, 0.25, 0.6}, Fr[3] = {0.0024, 0.0050, 0.0076}, Ro = 0.025;
    double idh0[4] = {0}, idh1[4] = {0}, s[3], t0[4] = {0}, t1[4], t2[4] = {0};
    for (int l = 0; l < 3; l++) { const double dhc = 0.5 * (dh[l] + dh[l + 1]); idh1[l] = 1. / (dhc * dh[l]); idh0[l + 1] = 1. / (dhc * dh[l + 1]); s[l] = (Fr[l] / Ro) * (Fr[l] / Ro); }
    for (int l = 0; l < 4; l++) { if (l > 0) t0[l] = -Delta * Delta * s[l - 1] * idh0[l]; if (l < 3) t2[l] = -Delta * Delta * s[l] * idh1[l]; t1[l] = -t0[l] - t2[l] + 4.; }
    for (int l = 1; l < 4; l++) t1[l] -= t0[l] * t2[l - 1] / t1[l - 1];
    for (int l = 0; l < 4; l++) { C.t0[l] = t0[l]; C.t2[l] = t2[l]; C.t1p[l] = t1[l]; C.rinv[l] = 1. / t1[l]; }
    for (int l = 0; l < 4; l++) { C.cf[l] = l > 0 ? t0[l] * C.rinv[l - 1] : 0.; C.cb[l] = t2[l] * C.rinv[l]; }
    C.msd2 = -Delta * Delta;
  }
  const size_t nd = g.plane * NL;
  std::vector<double> h(nd), hr(nd);
  srand(3);
  for (size_t i = 0; i < nd; i++) { h[i] = 1e-3 * (2.0 * rand() / RAND_MAX - 1.0); hr[i] = 2.0 * rand() / RAND_MAX - 1.0; }
  double *da, *res; int *err; long long *dbg; unsigned long long *mail;
  const int nworkers = (n + K - 1 + Cfg::W - 1) / Cfg::W;
  const size_t words = (size_t)nworkers * K * n * Cfg::NLP;
  CKC(cudaMalloc(&da, nd * 8)); CKC(cudaMalloc(&res, nd * 8)); CKC(cudaMalloc(&err, 4)); CKC(cudaMalloc(&dbg, (size_t)nworkers * 12 * 8));
  CKC(cudaMalloc(&mail, words * 8));
  CKC(cudaMemcpy(res, hr.data(), nd * 8, cudaMemcpyHostToDevice));
  CKC(cudaMemset(err, 0, 4));
  k_fill<<<592, 256>>>(mail, words, MAIL_EMPTY);
  RelaxArgs A;
  A.da = da; A.res = res; A.g = g; A.nsweeps = nsw; A.mailbox = mail; A.err = err; A.dbg = dbg; A.w_base = 0;
  constexpr int NTHR = 64 * BWPC;
  auto kern = k_relax_ws<NL, K, BWPC, false, false>;
  const size_t smem = Cfg::smem_per_worker * BWPC;
  CKC(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int mb = 0; CKC(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&mb, kern, NTHR, smem));
  const int grid = (nworkers + BWPC - 1) / BWPC;
  printf("n=%d nsweeps=%d workers=%d WPC=%d grid=%d smem/CTA=%zu B, CTAs/SM=%d\n", n, nsw, nworkers, BWPC, grid, smem, mb);
  if (grid > mb * 148) { printf("does not fit\n"); return 1; }
  void *args[] = {(void *)&A, (void *)&C};
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  float ms = 0;
  for (int rep = 0; rep < 3; rep++) {
    CKC(cudaMemcpy(da, h.data(), nd * 8, cudaMemcpyHostToDevice));
    CKC(cudaDeviceSynchronize());
    cudaEventRecord(e0);
    CKC(cudaLaunchCooperativeKernel((void *)kern, dim3(grid), dim3(NTHR), args, smem, 0));
    cudaEventRecord(e1);
    CKC(cudaDeviceSynchronize());
    cudaEventElapsedTime(&ms, e0, e1);
  }
  int herr; CKC(cudaMemcpy(&herr, err, 4, cudaMemcpyDeviceToHost));
  std::vector<long long> d((size_t)nworkers * 4);
  CKC(cudaMemcpy(d.data(), dbg, d.size() * 8, cudaMemcpyDeviceToHost));
  std::vector<double> o(nd);
  CKC(cudaMemcpy(o.data(), da, nd * 8, cudaMemcpyDeviceToHost));
  unsigned long long cs = 0;
  for (int l = 0; l < NL; l++) for (int y = 0; y < n; y++) for (int x = 0; x < n; x++) {
    unsigned long long u; double v = o[l * g.plane + GIDX(g.pitch, y, x)]; memcpy(&u, &v, 8); cs = cs * 1000003ull + u;
  }
  long long t0 = d[0]; for (int w = 0; w < nworkers; w++) t0 = std::min(t0, d[w * 4]);
  std::vector<double> lag;
  for (int w = 1; w < nworkers; w++) lag.push_back((d[w * 4 + 1] - d[(w - 1) * 4 + 1]) / 1e3);
  std::sort(lag.begin(), lag.end());
  const int steps = n + Cfg::W + 2 * K - 1;
  printf("kernel %.3f ms (err %d) | worker0 %.4f us/step (%.0f cycles @1.965GHz) | end-lag median %.3f us -> handoff %.3f us | checksum %016llx\n",
         ms, herr, (d[1] - d[0]) / 1e3 / steps, (d[1] - d[0]) / 1e3 / steps * 1965, lag[lag.size() / 2],
         lag[lag.size() / 2] - Cfg::W * (d[1] - d[0]) / 1e3 / steps, cs);
  // determinism stress: the strips synchronise through counters and self-validating mailbox entries only; repeat
  // the launch and compare the result bit for bit (argv[3] = repetitions)
  const int reps = argc > 3 ? atoi(argv[3]) : 0;
  int bad = 0;
  for (int r = 0; r < reps; r++) {
    CKC(cudaMemcpy(da, h.data(), nd * 8, cudaMemcpyHostToDevice));
    CKC(cudaLaunchCooperativeKernel((void *)kern, dim3(grid), dim3(NTHR), args, smem, 0));
    CKC(cudaDeviceSynchronize());
    std::vector<double> o2(nd);
    CKC(cudaMemcpy(o2.data(), da, nd * 8, cudaMemcpyDeviceToHost));
    if (memcmp(o2.data(), o.data(), nd * 8) != 0) bad++;
    CKC(cudaMemcpy(&herr, err, 4, cudaMemcpyDeviceToHost));
    if (herr) { printf("err flag %d at repetition %d\n", herr, r); break; }
  }
  if (reps) printf("determinism: %d of %d repetitions differ from the first result\n", bad, reps);
  for (int w : {0, 1, 2, 3, 4, nworkers / 2, nworkers - 2, nworkers - 1})
    printf("  w=%4d dur %8.1f us  spins %8lld  helper iters %8lld (%.3f us/iter)\n", w, (d[w * 4 + 1] - d[w * 4]) / 1e3, d[w * 4 + 2], d[w * 4 + 3],
           (d[w * 4 + 1] - d[w * 4]) / 1e3 / (double)std::max(1ll, d[w * 4 + 3]));
  return 0;
}
