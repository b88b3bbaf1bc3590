// TEST-ONLY device harness: the PTX carry-chain primitives of fp.cuh, the lazily reduced Granger-Scott squaring, the
// in-place Fp12 operations on a shared-memory slot and the two-lane operations of pairing_lanes.cuh, on RAW Montgomery
// limbs so that the tests can place values exactly at the bounds the source comments state.  The device twin of
// lazy_fp4.cu (which runs the host versions).  Never part of libsylow_b200.so; used by tests/test_gpu_device_bounds.py.
// Device memory and the stream come from the caller; the launchers allocate and copy nothing and do not synchronise.
#include "../../sylow_b200/csrc/pairing_lanes.cuh"
#include "../../sylow_b200/csrc/wire.cuh"

using namespace sylow;

// The kernels' shared-memory strides (kernels_pairing.cuh: SY_ACC_STRIDE, SY_SLOT_STRIDE, SY_FHOT_STRIDE).  That
// header is not included because it would compile the four pairing kernels into this harness as well.
#define DB_ACC_STRIDE 400
#define DB_SLOT_STRIDE 1040
#define DB_FHOT_STRIDE 784
#define DB_THREADS 64  // 64 slots of 400 bytes or 32 lane pairs of 1 040 bytes: below the 48 KB default

// ---- primitives: 64 input words and 32 output words per item (unused output words stay as the caller set them)
enum Prim {
  P_MUL_WIDE,     // r[0..16] = a[0..8] * a[8..16]
  P_REDC_WIDE,    // r[0..8] = fp_redc_wide(a[0..16])
  P_REDC_LOW,     // r[0..8] = redc_low(a[0..8])
  P_MUL,          // r[0..8] = fp_mul(a[0..8], a[8..16])
  P_FP2_MUL,      // r[0..16] = fp2_mul(a[0..16], a[16..32])
  P_WIDE_SUB,     // r[0..16] = a[0..16] - a[16..32] mod 2^512, r[16] = the borrow mask
  P_WIDE_ADD_PR,  // r[0..16] = wide_add_pR(a[0..16], mask a[16])
  P_LIFT_SUB1,    // r[0..17] = acc_lift_sub(p, a[0..16])
  P_LIFT_SUB2,    // r[0..17] = acc_lift_sub(2p, a[0..16])
  P_ACC_ADD,      // r[0..17] = a[0..17] + a[17..33]
  P_ACC_SUB,      // r[0..17] = a[0..17] - a[17..33]
  P_ACC_MADD9,    // r[0..17] = a[0..17] + 9 a[17..33]
  P_REDC_ACC,     // r[0..9] = fp_redc_acc(a[0..17])
  P_LIN9_ACC,     // r[0..9] = a[0..9] + a[9..17]
  P_LIN9_REDUCE,  // r[0..8] = lin9_reduce(a[0..9])
  P_U9_SHL0,      // r[0..9] = u9_add_shl(a[0..9], a[9..18], 0)
  P_U9_SHL1,      //                                         1
  P_U9_SHL3,      //                                         3
  P_LIN3,         // r[0..8] = fp_lin3(a[0..9], a[9..17])
  P_GS,           // r[0..32] = the new (x, y) of gs_fp4_square(a, b, x, y, false), a[0..64] = a, b, x, y
  P_GS_XI,        //                                                    true
};

__device__ __forceinline__ Fp fp_at(const uint32_t* a) {
  Fp r;
#pragma unroll
  for (int k = 0; k < 8; k++) r.l[k] = a[k];
  return r;
}
__device__ __forceinline__ void put(uint32_t* r, const Fp& x) {
#pragma unroll
  for (int k = 0; k < 8; k++) r[k] = x.l[k];
}

__global__ void k_prim(int op, const uint32_t* __restrict__ in, uint32_t* __restrict__ out, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t a[64], r[32];
#pragma unroll
  for (int k = 0; k < 64; k++) a[k] = in[64 * i + k];
#pragma unroll
  for (int k = 0; k < 32; k++) r[k] = out[32 * i + k];
  uint32_t p1[8], p2[8];
#pragma unroll
  for (int k = 0; k < 8; k++) {
    p1[k] = SY_TAB(kP)[k];
    p2[k] = SY_TAB(kP2)[k];
  }
  switch (op) {
    case P_MUL_WIDE: fp_mul_wide(r, a, a + 8); break;
    case P_REDC_WIDE: put(r, fp_redc_wide(a)); break;
#if defined(__CUDA_ARCH__)  // device only: the host build has no separate low-half reduction
    case P_REDC_LOW: put(r, redc_low(a)); break;
#endif
    case P_MUL: put(r, fp_mul(fp_at(a), fp_at(a + 8))); break;
    case P_FP2_MUL: {
      Fp2 x{fp_at(a), fp_at(a + 8)}, y{fp_at(a + 16), fp_at(a + 24)};
      Fp2 z = fp2_mul(x, y);
      put(r, z.c0);
      put(r + 8, z.c1);
    } break;
    case P_WIDE_SUB:
#pragma unroll
      for (int k = 0; k < 16; k++) r[k] = a[k];
      r[16] = wide_sub(r, a + 16);
      break;
    case P_WIDE_ADD_PR:
#pragma unroll
      for (int k = 0; k < 16; k++) r[k] = a[k];
      wide_add_pR(r, a[16]);
      break;
    case P_LIFT_SUB1: acc_lift_sub(r, p1, a); break;
    case P_LIFT_SUB2: acc_lift_sub(r, p2, a); break;
    case P_ACC_ADD:
    case P_ACC_SUB:
    case P_ACC_MADD9:
#pragma unroll
      for (int k = 0; k < 17; k++) r[k] = a[k];
      if (op == P_ACC_ADD) acc_add(r, a + 17);
      else if (op == P_ACC_SUB) acc_sub(r, a + 17);
      else acc_madd<9>(r, a + 17);
      break;
    case P_REDC_ACC: fp_redc_acc(r, a); break;
    case P_LIN9_ACC:
#pragma unroll
      for (int k = 0; k < 9; k++) r[k] = a[k];
      lin9_acc(r, a + 9);
      break;
    case P_LIN9_REDUCE: put(r, lin9_reduce(a)); break;
    case P_U9_SHL0: u9_add_shl(r, a, a + 9, 0); break;
    case P_U9_SHL1: u9_add_shl(r, a, a + 9, 1); break;
    case P_U9_SHL3: u9_add_shl(r, a, a + 9, 3); break;
    case P_LIN3: put(r, fp_lin3(a, fp_at(a + 9))); break;
    case P_GS:
    case P_GS_XI: {
      Fp2 v[4];
#pragma unroll
      for (int k = 0; k < 4; k++) v[k] = Fp2{fp_at(a + 16 * k), fp_at(a + 16 * k + 8)};
      gs_fp4_square(v[0], v[1], v[2], v[3], op == P_GS_XI);
      put(r, v[2].c0);
      put(r + 8, v[2].c1);
      put(r + 16, v[3].c0);
      put(r + 24, v[3].c1);
    } break;
  }
#pragma unroll
  for (int k = 0; k < 32; k++) out[32 * i + k] = r[k];
}

// ---- the in-place Fp12 operations where the kernels keep them: f in a shared-memory slot as k_miller / k_final_exp
enum Slot { S_SQR, S_SPARSE, S_CYCLOTOMIC, S_MUL, S_MUL_CONJ };

extern __shared__ uint4 db_smem[];

// out[i] = op(a[i], b[i]), 384-byte raw Fp12 values; the sparse factor is (b.c0.c0, b.c0.c1, b.c0.c2) = (l0, l_vw, l_vv)
__global__ void k_fp12_slot(int op, const uint8_t* a, const uint8_t* b, uint8_t* out, int n) {
  int i0 = blockIdx.x * blockDim.x + threadIdx.x;
  int i = i0 < n ? i0 : n - 1;  // as the kernels: every thread runs, the surplus is discarded
  Fp12& f = *reinterpret_cast<Fp12*>(reinterpret_cast<char*>(db_smem) + (size_t)threadIdx.x * DB_ACC_STRIDE);
  f = fp12_load_raw(a + 384 * i);
  const Fp12 g = fp12_load_raw(b + 384 * i);
  switch (op) {
    case S_SQR: fp12_sqr_assign(f); break;
    case S_SPARSE: fp12_sparse_mul_assign(f, g.c0.c0, g.c0.c1, g.c0.c2); break;
    case S_CYCLOTOMIC: cyclotomic_square_assign(f); break;
    case S_MUL: fp12_mul_assign(f, g, false); break;
    case S_MUL_CONJ: fp12_mul_assign(f, g, true); break;
  }
  if (i0 < n) fp12_store_raw(out + 384 * i, f);
}

// ---- the two-lane operations: thread 2k + role works on item k of the block, PairSlot / FexpHot in shared memory
enum Lanes { L_SQR, L_SPARSE, L_MUL, L_MUL_CONJ, L_CYCLOTOMIC, L_FROB1, L_FROB2, L_FROB3, L_INV };

__device__ __forceinline__ void load_half(Fp12& d, const uint8_t* p, int role) {
  const uint8_t* q = p + role * 192;
  Fp6 v{fp2_load_raw(q), fp2_load_raw(q + 64), fp2_load_raw(q + 128)};
  if (role) d.c1 = v;
  else d.c0 = v;
}

// out[i] = op(a[i], b[i]) as k_fp12_slot.  The second factor, the Frobenius and inverse inputs are read in place from
// global memory (k_final_exp_lanes reads them from its global FexpCold record).  SY_LANE_SYNC is __syncwarp(), so every
// thread runs the operation: surplus lane pairs redo the last item and discard it.
__global__ void k_lanes(int op, const uint8_t* a, const uint8_t* b, uint8_t* out, int n) {
  const int role = threadIdx.x & 1;
  const unsigned slot = threadIdx.x >> 1;
  int i0 = blockIdx.x * (blockDim.x >> 1) + slot;
  int i = i0 < n ? i0 : n - 1;
  PairSlot& s = *reinterpret_cast<PairSlot*>(reinterpret_cast<char*>(db_smem) + (size_t)slot * DB_SLOT_STRIDE);
  FexpHot& h = *reinterpret_cast<FexpHot*>(reinterpret_cast<char*>(db_smem) + (size_t)slot * DB_FHOT_STRIDE);
  const Fp12& A = *reinterpret_cast<const Fp12*>(a + 384 * i);
  const Fp12& B = *reinterpret_cast<const Fp12*>(b + 384 * i);
  Fp12* res = &h.res;
  switch (op) {
    case L_SQR:
    case L_SPARSE:
      load_half(s.f, a + 384 * i, role);
      if (!role) s.l = Ell{fp2_load_raw(b + 384 * i), fp2_load_raw(b + 384 * i + 64), fp2_load_raw(b + 384 * i + 128)};
      SY_LANE_SYNC();
      if (op == L_SQR) lanes_fp12_sqr(s, role);
      else lanes_sparse_mul(s, role);
      res = &s.f;
      break;
    case L_MUL:
    case L_MUL_CONJ:
    case L_CYCLOTOMIC:
      load_half(h.res, a + 384 * i, role);
      SY_LANE_SYNC();
      if (op == L_CYCLOTOMIC) lanes_cyclotomic_square(h.x, h.res, role);
      else lanes_fp12_mul(h.x, h.res, B, op == L_MUL_CONJ, role);
      break;
    case L_FROB1:
    case L_FROB2:
    case L_FROB3: lanes_frobenius_to(h.res, A, op - L_FROB1 + 1, role); break;
    case L_INV: lanes_fp12_inv(h.x, h.res, A, role); break;
  }
  if (i0 >= n) return;
  // lane 0 stores c0, lane 1 stores c1 (every operation ends with a lane-pair barrier)
  const Fp6& r = role ? res->c1 : res->c0;
  uint8_t* o = out + 384 * i + role * 192;
  fp2_store_raw(o, r.c0);
  fp2_store_raw(o + 64, r.c1);
  fp2_store_raw(o + 128, r.c2);
}

extern "C" {

int db_prim(int op, const void* in, void* out, int n, void* stream) {
  if (n <= 0) return 0;
  k_prim<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(op, (const uint32_t*)in, (uint32_t*)out, n);
  return (int)cudaGetLastError();
}

int db_fp12_slot(int op, const void* a, const void* b, void* out, int n, void* stream) {
  if (n <= 0) return 0;
  k_fp12_slot<<<(n + DB_THREADS - 1) / DB_THREADS, DB_THREADS, DB_THREADS * DB_ACC_STRIDE, (cudaStream_t)stream>>>(
      op, (const uint8_t*)a, (const uint8_t*)b, (uint8_t*)out, n);
  return (int)cudaGetLastError();
}

int db_lanes(int op, const void* a, const void* b, void* out, int n, void* stream) {
  if (n <= 0) return 0;
  const int pairs = DB_THREADS / 2;
  k_lanes<<<(n + pairs - 1) / pairs, DB_THREADS, pairs * DB_SLOT_STRIDE, (cudaStream_t)stream>>>(
      op, (const uint8_t*)a, (const uint8_t*)b, (uint8_t*)out, n);
  return (int)cudaGetLastError();
}

}  // extern "C"
