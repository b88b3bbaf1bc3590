// The two kernels of the pairing step (BASELINE configs[1]): k_miller and k_final_exp, with their launch shapes.
// Kept in a header so that the library (sylow_b200.cu) and the stand-alone timing harness (tools/kbench.cu) compile
// exactly the same code.
#pragma once
#include "wire.cuh"
#include "pairing_lanes.cuh"

#define SY_MILLER_THREADS 128
// Three 128-thread blocks per SM at 168 registers run one plain launch of 2^20 pairs 1 % faster (164.4 against 166.2 ms,
// profiles/r02h_kbench.jsonl) but lose it again in the library, where the wave remainders run at low occupancy
// (2^20: 167.6 against 166.0 ms, 2^17: 22.3 against 21.6 ms, profiles/r02i_policy_sweep_m128x3.jsonl): two blocks stay.
#define SY_MILLER_MINB 2
#define SY_GLUED_THREADS 128
#define SY_GLUED_MINB 2
#define SY_FEXP_THREADS 384
#define SY_FEXP_MINB 1

// Shared-memory slot of one thread's hot Fp12 accumulator: 384 bytes padded to 400, so that the eight lanes of a
// 128-bit shared-memory access phase fall into different banks (100 words x lane = 4 x lane mod 32).
// Measured at 2^20 (profiles/r02_kbench_*.jsonl): the Miller loop with its accumulator f in shared memory 170.0 ->
// 166.1 ms (and no register spills left); the Miller loop's G2 point in shared memory as well: slower (169.6).  The final
// exponentiation's running value in shared memory made no difference while the Granger-Scott squaring still copied it
// (174.6 / 174.7 ms); with the in-place squaring it does: 160.6 -> 158.1 ms (profiles/r02v_kbench_fexp_smem.jsonl).
#define SY_ACC_STRIDE 400
// Two lanes per Miller loop (pairing_lanes.cuh): one PairSlot (1 024 bytes) per lane pair, padded to 1 040 so that
// consecutive slots start four banks apart (the eight lanes of a 128-bit access phase are four pairs).
#define SY_LANES_THREADS 128
#define SY_LANES_MINB 2
#define SY_SLOT_STRIDE 1040
#define SY_LANES_SMEM_BYTES(threads) ((size_t)((threads) / 2) * SY_SLOT_STRIDE)
// two lanes per final exponentiation: FexpHot (768 bytes) per lane pair, padded the same way; FexpCold in global scratch
#define SY_FHOT_STRIDE 784
#define SY_FLANES_SMEM_BYTES(threads) ((size_t)((threads) / 2) * SY_FHOT_STRIDE)
#define SY_FLANES_SCRATCH_BYTES(pairs) ((size_t)(pairs) * sizeof(sylow::FexpCold))
#define SY_MILLER_SMEM_BYTES(threads) ((size_t)(threads) * SY_ACC_STRIDE)
#define SY_FEXP_SMEM_BYTES(threads) ((size_t)(threads) * SY_ACC_STRIDE)

namespace sylow_kernels {
using namespace sylow;
extern __shared__ uint4 sy_acc_smem[];
__device__ __forceinline__ Fp12* acc_slot() {
  return reinterpret_cast<Fp12*>(reinterpret_cast<char*>(sy_acc_smem) + (size_t)threadIdx.x * SY_ACC_STRIDE);
}

// f_out[i] = miller_loop(g2[i * g2_stride], g1[i]) (Montgomery form if raw_out, else canonical).
__global__ void __launch_bounds__(SY_MILLER_THREADS, SY_MILLER_MINB)
k_miller(const uint8_t* __restrict__ g1, const uint8_t* __restrict__ g1_inf, const uint8_t* __restrict__ g2,
         const uint8_t* __restrict__ g2_inf, size_t g2_stride, size_t n, uint8_t* __restrict__ f_out, int raw_out) {
  size_t i0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  // Every thread of the block runs the loop (SY_LOOP_SYNC needs that): out-of-range threads redo the
  // last item and discard it; infinite pairs are computed on whatever bytes are there and replaced by 1.
  size_t i = i0 < n ? i0 : n - 1;
  size_t j = i * g2_stride;
  bool inf = (g1_inf && g1_inf[i]) || (g2_inf && g2_inf[j]);
  const uint8_t* p = g1 + i * 64;
  const uint8_t* q = g2 + j * 128;
  Fp12 f = miller_loop(fp_load(p), fp_load(p + 32), fp2_load(q), fp2_load(q + 64), acc_slot());
  if (i0 >= n) return;
  if (inf) f = fp12_one();
  if (raw_out)
    fp12_store_raw(f_out + i * 384, f);
  else
    fp12_store(f_out + i * 384, f);
}

// The same values as k_miller with two lanes per pair: thread 2k + role of a block works on pair k of the block.
__global__ void __launch_bounds__(SY_LANES_THREADS, SY_LANES_MINB)
k_miller_lanes(const uint8_t* __restrict__ g1, const uint8_t* __restrict__ g1_inf, const uint8_t* __restrict__ g2,
               const uint8_t* __restrict__ g2_inf, size_t n, uint8_t* __restrict__ f_out, int raw_out) {
  const int role = threadIdx.x & 1;
  const unsigned slot = threadIdx.x >> 1;
  size_t i0 = (size_t)blockIdx.x * (blockDim.x >> 1) + slot;
  size_t i = i0 < n ? i0 : n - 1;  // surplus lane pairs redo the last item (every thread runs the loop)
  bool inf = (g1_inf && g1_inf[i]) || (g2_inf && g2_inf[i]);
  const uint8_t* p = g1 + i * 64;
  const uint8_t* q = g2 + i * 128;
  PairSlot& s = *reinterpret_cast<PairSlot*>(reinterpret_cast<char*>(sy_acc_smem) + (size_t)slot * SY_SLOT_STRIDE);
  lanes_miller_loop(s, role, fp_load(p), fp_load(p + 32), fp2_load(q), fp2_load(q + 64));
  if (i0 >= n) return;
  // lane 0 stores c0, lane 1 stores c1
  Fp6 h = role ? s.f.c1 : s.f.c0;
  if (inf) h = role ? fp6_zero() : fp6_one();
  uint8_t* o = f_out + i * 384 + role * 192;
  if (raw_out) {
    fp2_store_raw(o, h.c0);
    fp2_store_raw(o + 64, h.c1);
    fp2_store_raw(o + 128, h.c2);
  } else {
    fp2_store(o, h.c0);
    fp2_store(o + 64, h.c1);
    fp2_store(o + 128, h.c2);
  }
}

__global__ void __launch_bounds__(SY_FEXP_THREADS, SY_FEXP_MINB)
k_final_exp(const uint8_t* f_in, int raw_in, size_t n, uint8_t* gt_out) {
  size_t i0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t i = i0 < n ? i0 : n - 1;  // all threads run the loops (SY_LOOP_SYNC); the surplus is discarded
  Fp12 f = raw_in ? fp12_load_raw(f_in + i * 384) : fp12_load(f_in + i * 384);
  final_exponentiation_assign(f, acc_slot());
  if (i0 >= n) return;
  fp12_store(gt_out + i * 384, f);
}

// The same values as k_final_exp with two lanes per item.  `scratch` holds one FexpCold per launched lane pair
// (gridDim.x * blockDim.x / 2 of them).
__global__ void __launch_bounds__(SY_LANES_THREADS, SY_LANES_MINB)
k_final_exp_lanes(const uint8_t* f_in, int raw_in, size_t n, uint8_t* gt_out, uint8_t* scratch) {
  const int role = threadIdx.x & 1;
  const unsigned slot = threadIdx.x >> 1;
  size_t i0 = (size_t)blockIdx.x * (blockDim.x >> 1) + slot;
  size_t i = i0 < n ? i0 : n - 1;
  FexpHot& h = *reinterpret_cast<FexpHot*>(reinterpret_cast<char*>(sy_acc_smem) + (size_t)slot * SY_FHOT_STRIDE);
  FexpCold& c = reinterpret_cast<FexpCold*>(scratch)[i0];
  const uint8_t* p = f_in + i * 384 + role * 192;
  Fp6 v;
  if (raw_in)
    v = Fp6{fp2_load_raw(p), fp2_load_raw(p + 64), fp2_load_raw(p + 128)};
  else
    v = Fp6{fp2_load(p), fp2_load(p + 64), fp2_load(p + 128)};
  if (role) c.f.c1 = v;
  else c.f.c0 = v;
  SY_LANE_SYNC();
  lanes_final_exponentiation(h, c, role);
  if (i0 >= n) return;
  const Fp6& r = role ? c.E.c1 : c.E.c0;
  uint8_t* o = gt_out + i * 384 + role * 192;
  fp2_store(o, r.c0);
  fp2_store(o + 64, r.c1);
  fp2_store(o + 128, r.c2);
}

}  // namespace sylow_kernels
using namespace sylow_kernels;
