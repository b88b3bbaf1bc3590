// Stand-alone timing + checksum harness for the two pairing kernels (k_miller, k_final_exp), compiled from the SAME
// header as the library (csrc/kernels_pairing.cuh).  Used to compare the kernels of two checkouts (tools/kbench_build.sh
// name:tree ...) on the GPU without the 3-minute full-library build: every variant prints its kernel times and a
// checksum of the outputs on fixed pseudo-random inputs, so a variant that changes a single bit of any result is caught
// in the same run.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -DSY_VARIANT='"name"' \
//        -o build/kbench/name tools/kbench.cu
//   build/kbench/name [log2n=18] [reps=3] [n=2^log2n] [miller block threads] [lanes block threads]
// The two-lane Miller kernel (k_miller_lanes) runs on the same inputs and must give the same checksum as k_miller.
// Inputs are arbitrary field elements (not curve points): both kernels are branch-free in the data, and the parity
// of the real thing is the job of tests/ (this tool only says "same bits as the baseline variant, and how fast").
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>

#include "../sylow_b200/csrc/kernels_pairing.cuh"

#ifndef SY_VARIANT
#define SY_VARIANT "base"
#endif

__global__ void k_fill(uint32_t* p, size_t words, uint64_t seed) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= words) return;
  uint64_t z = seed + 0x9e3779b97f4a7c15ull * (i + 1);
  z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
  z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
  z ^= z >> 31;
  uint32_t v = (uint32_t)z;
  if ((i & 7) == 7) v &= 0x1fffffffu;  // keep every 32-byte value below 2^253 < p
  p[i] = v;
}
__global__ void k_checksum(const uint32_t* p, size_t words, unsigned long long* out) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long v = 0;
  for (; i < words; i += (size_t)gridDim.x * blockDim.x) v += (unsigned long long)p[i] * (2 * (i % 1000003) + 1);
  atomicAdd(out, v);
}
#define CHECK(x)                                                                  \
  do {                                                                            \
    cudaError_t e = (x);                                                          \
    if (e != cudaSuccess) {                                                       \
      fprintf(stderr, "%s:%d %s\n", __FILE__, __LINE__, cudaGetErrorString(e));   \
      return 1;                                                                   \
    }                                                                             \
  } while (0)

static unsigned long long checksum(const uint8_t* d, size_t bytes, unsigned long long* d_sum) {
  cudaMemset(d_sum, 0, 8);
  k_checksum<<<1024, 256>>>((const uint32_t*)d, bytes / 4, d_sum);
  unsigned long long h = 0;
  cudaMemcpy(&h, d_sum, 8, cudaMemcpyDeviceToHost);
  return h;
}

int main(int argc, char** argv) {
  int log2n = argc > 1 ? atoi(argv[1]) : 18;
  int reps = argc > 2 ? atoi(argv[2]) : 3;
  size_t n = argc > 3 && atol(argv[3]) > 0 ? (size_t)atol(argv[3]) : (size_t)1 << log2n;
  int mt = argc > 4 ? atoi(argv[4]) : SY_MILLER_THREADS;
  int lt = argc > 5 ? atoi(argv[5]) : SY_LANES_THREADS;
  uint8_t *g1, *g2, *f, *gt;
  unsigned long long* d_sum;
  CHECK(cudaMalloc(&g1, n * 64));
  CHECK(cudaMalloc(&g2, n * 128));
  CHECK(cudaMalloc(&f, n * 384));
  CHECK(cudaMalloc(&gt, n * 384));
  CHECK(cudaMalloc(&d_sum, 8));
  k_fill<<<(unsigned)((n * 16 + 255) / 256), 256>>>((uint32_t*)g1, n * 16, 1);
  k_fill<<<(unsigned)((n * 32 + 255) / 256), 256>>>((uint32_t*)g2, n * 32, 2);
  CHECK(cudaDeviceSynchronize());
  cudaEvent_t a, b;
  cudaEventCreate(&a);
  cudaEventCreate(&b);
  float ms_m = 0, ms_f = 0;
  unsigned gm = (unsigned)((n + mt - 1) / mt);
  unsigned gl = (unsigned)((n + lt / 2 - 1) / (lt / 2));
  float ms_l = 0;
  unsigned gf = (unsigned)((n + SY_FEXP_THREADS - 1) / SY_FEXP_THREADS);
  const size_t sm_m = SY_MILLER_SMEM_BYTES(mt);
  const size_t sm_l = SY_LANES_SMEM_BYTES(lt);
  CHECK(cudaFuncSetAttribute(k_miller, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)SY_MILLER_SMEM_BYTES(SY_MILLER_THREADS)));
  CHECK(cudaFuncSetAttribute(k_miller_lanes, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)SY_LANES_SMEM_BYTES(SY_LANES_THREADS)));
  const size_t sm_f = SY_FEXP_SMEM_BYTES(SY_FEXP_THREADS);
  CHECK(cudaFuncSetAttribute(k_final_exp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_f));
  k_miller_lanes<<<gl, lt, sm_l>>>(g1, nullptr, g2, nullptr, n, f, 1);
  CHECK(cudaDeviceSynchronize());
  cudaEventRecord(a);
  for (int r = 0; r < reps; r++) k_miller_lanes<<<gl, lt, sm_l>>>(g1, nullptr, g2, nullptr, n, f, 1);
  cudaEventRecord(b);
  CHECK(cudaDeviceSynchronize());
  cudaEventElapsedTime(&ms_l, a, b);
  unsigned long long cl = checksum(f, n * 384, d_sum);
  CHECK(cudaMemset(f, 0, n * 384));
  k_miller<<<gm, mt, sm_m>>>(g1, nullptr, g2, nullptr, 1, n, f, 1);
  CHECK(cudaDeviceSynchronize());
  cudaEventRecord(a);
  for (int r = 0; r < reps; r++) k_miller<<<gm, mt, sm_m>>>(g1, nullptr, g2, nullptr, 1, n, f, 1);
  cudaEventRecord(b);
  CHECK(cudaDeviceSynchronize());
  cudaEventElapsedTime(&ms_m, a, b);
  unsigned long long cm = checksum(f, n * 384, d_sum);
  k_final_exp<<<gf, SY_FEXP_THREADS, sm_f>>>(f, 1, n, gt);
  CHECK(cudaDeviceSynchronize());
  cudaEventRecord(a);
  for (int r = 0; r < reps; r++) k_final_exp<<<gf, SY_FEXP_THREADS, sm_f>>>(f, 1, n, gt);
  cudaEventRecord(b);
  CHECK(cudaDeviceSynchronize());
  cudaEventElapsedTime(&ms_f, a, b);
  unsigned long long cf = checksum(gt, n * 384, d_sum);
  // two lanes per final exponentiation
  uint8_t* fscr;
  float ms_fl = 0;
  CHECK(cudaMalloc(&fscr, SY_FLANES_SCRATCH_BYTES((size_t)gl * (lt / 2))));
  CHECK(cudaFuncSetAttribute(k_final_exp_lanes, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)SY_FLANES_SMEM_BYTES(SY_LANES_THREADS)));
  CHECK(cudaMemset(gt, 0, n * 384));
  k_final_exp_lanes<<<gl, lt, SY_FLANES_SMEM_BYTES(lt)>>>(f, 1, n, gt, fscr);
  CHECK(cudaDeviceSynchronize());
  cudaEventRecord(a);
  for (int r = 0; r < reps; r++) k_final_exp_lanes<<<gl, lt, SY_FLANES_SMEM_BYTES(lt)>>>(f, 1, n, gt, fscr);
  cudaEventRecord(b);
  CHECK(cudaDeviceSynchronize());
  cudaEventElapsedTime(&ms_fl, a, b);
  unsigned long long cfl = checksum(gt, n * 384, d_sum);
  cudaFuncAttributes afl;
  cudaFuncGetAttributes(&afl, k_final_exp_lanes);
  cudaFuncAttributes am, af, al;
  cudaFuncGetAttributes(&al, k_miller_lanes);
  cudaFuncGetAttributes(&am, k_miller);
  cudaFuncGetAttributes(&af, k_final_exp);
  printf("{\"variant\": \"%s\", \"n\": %zu, \"miller_threads\": %d, \"lanes_threads\": %d, \"ms_lanes\": %.3f, "
         "\"sum_lanes\": \"%016llx\", \"lanes_regs\": %d, \"lanes_frame\": %zu, \"lanes_match\": %s, ",
         SY_VARIANT, n, mt, lt, ms_l / reps, cl, al.numRegs, al.localSizeBytes, cl == cm ? "true" : "false");
  printf("\"ms_fexp_lanes\": %.3f, \"fexp_lanes_match\": %s, \"fexp_lanes_regs\": %d, \"fexp_lanes_frame\": %zu, ",
         ms_fl / reps, cfl == cf ? "true" : "false", afl.numRegs, afl.localSizeBytes);
  printf("\"log2n\": %d, \"ms_miller\": %.3f, \"ms_fexp\": %.3f, \"pairings_per_s\": %.0f, "
         "\"sum_miller\": \"%016llx\", \"sum_fexp\": \"%016llx\", \"miller_regs\": %d, \"miller_frame\": %zu, "
         "\"fexp_regs\": %d, \"fexp_frame\": %zu}\n",
         log2n, ms_m / reps, ms_f / reps, n / ((ms_m + ms_f) / reps) * 1e3, cm, cf, am.numRegs,
         am.localSizeBytes, af.numRegs, af.localSizeBytes);
  return 0;
}
