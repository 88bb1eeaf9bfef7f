// See ewe.cuh.  All kernels are streaming (HBM-bound) except base conversion (FP64 tensor-core path, pipe bound).
#include "ewe.cuh"
#include "launch.h"

#include <algorithm>
#include <cstdlib>
#include <type_traits>

namespace hml {

constexpr int EW_THREADS = 256;  // 2 coefficients per thread, 16-byte accesses

__device__ __forceinline__ ulonglong2 ld2(const u64 *p, size_t i2) { return __ldg(reinterpret_cast<const ulonglong2 *>(p) + i2); }
__device__ __forceinline__ void st2(u64 *p, size_t i2, u64 a, u64 b) { reinterpret_cast<ulonglong2 *>(p)[i2] = make_ulonglong2(a, b); }
__device__ __forceinline__ u64 finish(double v, const ModConst &m) { return f64_to_canonical(reduce_signed(v, m.q, m.qinv), m.qi); }

static inline dim3 ew_grid(int N, int ny, int nz = 1) { return dim3((N / 2 + EW_THREADS - 1) / EW_THREADS, ny, nz); }

// ------------------------------------------------------------------------------------------------ generic EWE
// grid.z = component of a ciphertext op: operand k advances by cs[k] words per component (0 repeats a plaintext), out by cs[4]
struct EweStrides {
  long long cs[5];
};
__global__ void __launch_bounds__(EW_THREADS) k_ewe(const ModConst *__restrict__ mc, LimbMap lm, int N, const u64 *x1,
                                                    const u64 *x2, const u64 *x3, const u64 *x4, int subtract, u64 *out,
                                                    EweStrides st) {
  pdl_wait();
  const int i2 = blockIdx.x * EW_THREADS + threadIdx.x;
  if (i2 >= N / 2) return;
  const int limb = blockIdx.y;
  const ModConst m = mc[lm.mod[limb]];
  const size_t o = (size_t)limb * (N / 2) + i2;
  const long long z = blockIdx.z;
  if (x1) x1 += z * st.cs[0];
  if (x2) x2 += z * st.cs[1];
  if (x3) x3 += z * st.cs[2];
  if (x4) x4 += z * st.cs[3];
  out += z * st.cs[4];
  double p0 = 0, p1 = 0, s0 = 0, s1 = 0;
  if (x1) {
    ulonglong2 a = ld2(x1, o);
    p0 = u64_to_f64(a.x); p1 = u64_to_f64(a.y);
    if (x2) {
      ulonglong2 b = ld2(x2, o);
      p0 = mulmod_var(p0, u64_to_f64(b.x), m.q, m.qinv);
      p1 = mulmod_var(p1, u64_to_f64(b.y), m.q, m.qinv);
    }
  }
  if (x3) {
    ulonglong2 a = ld2(x3, o);
    s0 = u64_to_f64(a.x); s1 = u64_to_f64(a.y);
    if (x4) {
      ulonglong2 b = ld2(x4, o);
      s0 = mulmod_var(s0, u64_to_f64(b.x), m.q, m.qinv);
      s1 = mulmod_var(s1, u64_to_f64(b.y), m.q, m.qinv);
    }
  }
  if (subtract) { s0 = -s0; s1 = -s1; }
  st2(out, o, finish(p0 + s0, m), finish(p1 + s1, m));
}

void launch_ewe(const ModConst *mc, const LimbMap &lm, int N, int n_limbs, const u64 *x1, const u64 *x2, const u64 *x3,
                const u64 *x4, int subtract, u64 *out, cudaStream_t s, int n_comp, const long long *comp_strides) {
  EweStrides st{};
  if (comp_strides) for (int k = 0; k < 5; ++k) st.cs[k] = comp_strides[k];
  launch_pdl(k_ewe, ew_grid(N, n_limbs, n_comp), EW_THREADS, 0, s, mc, lm, N, x1, x2, x3, x4, subtract, out, st);
}

// ------------------------------------------------------------------------------------------------ tensor product
__global__ void __launch_bounds__(EW_THREADS) k_tensor3(const ModConst *__restrict__ mc, int N, const u64 *a0, const u64 *a1,
                                                        const u64 *b0, const u64 *b1, u64 *d0, u64 *d1, u64 *d2,
                                                        long long in_stride, long long out_stride, int pack01) {
  pdl_wait();
  const int i2 = blockIdx.x * EW_THREADS + threadIdx.x;
  if (i2 >= N / 2) return;
  const int limb = blockIdx.y;  // limbs 0..L-1 are moduli q_0..q_{L-1}
  const ModConst m = mc[limb];
  const size_t o = (size_t)limb * (N / 2) + i2;
  const long long bi = (long long)blockIdx.z * in_stride, bo = (long long)blockIdx.z * out_stride;  // ciphertext of the batch
  a0 += bi; a1 += bi; b0 += bi; b1 += bi; d0 += bo; d1 += bo; d2 += bo;
  const ulonglong2 A0 = ld2(a0, o), A1 = ld2(a1, o), B0 = ld2(b0, o), B1 = ld2(b1, o);
  u64 r0[2], r1[2], r2[2];
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const double x0 = u64_to_f64(k ? A0.y : A0.x), x1 = u64_to_f64(k ? A1.y : A1.x);
    const double y0 = u64_to_f64(k ? B0.y : B0.x), y1 = u64_to_f64(k ? B1.y : B1.x);
    r0[k] = f64_to_canonical(mulmod_var(x0, y0, m.q, m.qinv), m.qi);
    r1[k] = finish(mulmod_var(x0, y1, m.q, m.qinv) + mulmod_var(x1, y0, m.q, m.qinv), m);
    r2[k] = f64_to_canonical(mulmod_var(x1, y1, m.q, m.qinv), m.qi);
  }
  if (pack01) {
    st_packed2(d0 + (size_t)limb * N, N, i2, r0[0], r0[1]);
    st_packed2(d1 + (size_t)limb * N, N, i2, r1[0], r1[1]);
  } else {
    st2(d0, o, r0[0], r0[1]);
    st2(d1, o, r1[0], r1[1]);
  }
  st2(d2, o, r2[0], r2[1]);
}

void launch_tensor3(const ModConst *mc, int N, int L, const u64 *a0, const u64 *a1, const u64 *b0, const u64 *b1, u64 *d0,
                    u64 *d1, u64 *d2, int n_batch, long long in_stride, long long out_stride, cudaStream_t s, int pack01) {
  launch_pdl(k_tensor3, ew_grid(N, L, n_batch), EW_THREADS, 0, s, mc, N, a0, a1, b0, b1, d0, d1, d2, in_stride, out_stride, pack01);
}

// Sum of tensor products (ewe.cuh TensorSumArgs), k_tensor3's layout with a loop over the pairs; the pair table is read in place
// (grid constant).  The sums stay lazy doubles and each output is reduced once.  Exact: every mulmod_var product lies in
// (-0.51q, 0.51q), so with 16 pairs d1 sums 32 products plus one stored canonical word: |v| < 17.4q < 2^41 (q < 2^36), far
// inside reduce_signed's |v| < 2^51.
__global__ void __launch_bounds__(EW_THREADS) k_tensor_sum(const ModConst *__restrict__ mc, const __grid_constant__ TensorSumArgs a) {
  pdl_wait();
  const int i2 = blockIdx.x * EW_THREADS + threadIdx.x;
  if (i2 >= a.N / 2) return;
  const int limb = blockIdx.y;  // limb slot; its modulus is q_{mod0 + limb * mod_step}
  const ModConst m = mc[a.mod0 + limb * a.mod_step];
  const size_t o = (size_t)limb * (a.N / 2) + i2;
  const long long bi = (long long)blockIdx.z * a.in_stride, bo = (long long)blockIdx.z * a.out_stride;
  double s0[2] = {0, 0}, s1[2] = {0, 0}, s2[2] = {0, 0};
  for (int k = 0; k < a.n_pairs; ++k) {
    const u64 *pa = a.a[k] + bi, *pb = a.b[k] + bi;
    const ulonglong2 A0 = ld2(pa, o), A1 = ld2(pa + a.comp_stride, o);
    const bool sq = pa == pb;  // uniform: a square reads one ciphertext
    const ulonglong2 B0 = sq ? A0 : ld2(pb, o), B1 = sq ? A1 : ld2(pb + a.comp_stride, o);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const double x0 = u64_to_f64(h ? A0.y : A0.x), x1 = u64_to_f64(h ? A1.y : A1.x);
      const double y0 = u64_to_f64(h ? B0.y : B0.x), y1 = u64_to_f64(h ? B1.y : B1.x);
      s0[h] += mulmod_var(x0, y0, m.q, m.qinv);
      s1[h] += mulmod_var(x0, y1, m.q, m.qinv) + mulmod_var(x1, y0, m.q, m.qinv);
      s2[h] += mulmod_var(x1, y1, m.q, m.qinv);
    }
  }
  u64 *d0 = a.d0 + bo, *d1 = a.d1 + bo, *d2 = a.d2 + bo;
  if (a.accumulate) {  // uniform: a later group of the same op
    const ulonglong2 p0 = a.pack01 ? ld_packed2(d0 + (size_t)limb * a.N, a.N, i2) : ld2(d0, o);
    const ulonglong2 p1 = a.pack01 ? ld_packed2(d1 + (size_t)limb * a.N, a.N, i2) : ld2(d1, o);
    const ulonglong2 p2 = ld2(d2, o);
    s0[0] += u64_to_f64(p0.x); s0[1] += u64_to_f64(p0.y);
    s1[0] += u64_to_f64(p1.x); s1[1] += u64_to_f64(p1.y);
    s2[0] += u64_to_f64(p2.x); s2[1] += u64_to_f64(p2.y);
  }
  if (a.pack01) {
    st_packed2(d0 + (size_t)limb * a.N, a.N, i2, finish(s0[0], m), finish(s0[1], m));
    st_packed2(d1 + (size_t)limb * a.N, a.N, i2, finish(s1[0], m), finish(s1[1], m));
  } else {
    st2(d0, o, finish(s0[0], m), finish(s0[1], m));
    st2(d1, o, finish(s1[0], m), finish(s1[1], m));
  }
  st2(d2, o, finish(s2[0], m), finish(s2[1], m));
}

void launch_tensor_sum(const ModConst *mc, int L, int n_batch, const TensorSumArgs &a, cudaStream_t s) {
  launch_pdl(k_tensor_sum, ew_grid(a.N, L, n_batch), EW_THREADS, 0, s, mc, a);
}

// ------------------------------------------------------------------------------------------------ key-switch inner product
// The key words of a (limb, coefficient pair) are loaded once and reused for every ciphertext of the batch
// (the key is 60% of the traffic of an unbatched inner product).
// An empty asm statement that "uses" every loaded register: all the loads above it must have been ISSUED before any
// instruction below it (no instruction is emitted, so nothing waits here — the scoreboard stalls at the first real use).
#define HML_PIN4(v) "+l"(v[0].x), "+l"(v[0].y), "+l"(v[1].x), "+l"(v[1].y)
template <int NB>
__device__ __forceinline__ void pin_loads(ulonglong2 (&k)[NB][2]) {
  if constexpr (NB == 1) asm volatile("" : HML_PIN4(k[0]));
  else if constexpr (NB == 2) asm volatile("" : HML_PIN4(k[0]), HML_PIN4(k[1]));
  else if constexpr (NB == 3) asm volatile("" : HML_PIN4(k[0]), HML_PIN4(k[1]), HML_PIN4(k[2]));
  else if constexpr (NB == 4) asm volatile("" : HML_PIN4(k[0]), HML_PIN4(k[1]), HML_PIN4(k[2]), HML_PIN4(k[3]));
  else {
    asm volatile("" : HML_PIN4(k[0]), HML_PIN4(k[1]), HML_PIN4(k[2]), HML_PIN4(k[3]));
    asm volatile("" : HML_PIN4(k[4]), HML_PIN4(k[5]), HML_PIN4(k[6]), HML_PIN4(k[7]));
  }
}

// Source slots of coefficient pair i2 under the automorphism X -> X^g (g == 0: the identity): the slot k' the automorphism
// kernel would fetch, 2*brv(k')+1 = g*(2*brv(k)+1) mod 2N.
__device__ __forceinline__ uint2 gal_slots(unsigned g, int logN, int i2) {
  unsigned s0 = 2u * i2, s1 = 2u * i2 + 1u;
  if (g) {
    const unsigned sh = 32 - logN, m2n = (2u << logN) - 1u;
    s0 = __brev((((g * (2u * (__brev(s0) >> sh) + 1u)) & m2n) - 1u) >> 1) >> sh;
    s1 = __brev((((g * (2u * (__brev(s1) >> sh) + 1u)) & m2n) - 1u) >> 1) >> sh;
  }
  return make_uint2(s0, s1);
}
// coefficient pair i2 of a digit (or c0), read through the slots src when gal
__device__ __forceinline__ ulonglong2 ld_pair(const u64 *p, int i2, uint2 src, bool gal) {
  return gal ? make_ulonglong2(__ldg(p + src.x), __ldg(p + src.y)) : ld2(p, i2);
}
// The key words of digits j < beta at key limb kl (evk [beta][2][evk_limbs][N]; a = the kernel's argument struct, n2 = N / 2);
// padding digits are zero.  PACKED: the raw halves of packed limbs, joined by join_key after pin_loads.
template <bool PACKED, int NB, class A>
__device__ __forceinline__ void ld_key(ulonglong2 (&k)[NB][2], const u64 *evk, const A &a, int kl, size_t n2, int i2) {
#pragma unroll
  for (int j = 0; j < NB; ++j)
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      if constexpr (PACKED) {
        const u64 *slot = evk + (((size_t)j * 2 + c) * a.evk_limbs + kl) * a.N;
        k[j][c] = j < a.beta ? ld_packed2_raw(slot, a.N, i2) : make_ulonglong2(0, 0);
      } else {
        k[j][c] = j < a.beta ? ld2(evk, (((size_t)j * 2 + c) * a.evk_limbs + kl) * n2 + i2) : make_ulonglong2(0, 0);
      }
    }
}
template <int NB>
__device__ __forceinline__ void join_key(ulonglong2 (&k)[NB][2]) {
#pragma unroll
  for (int j = 0; j < NB; ++j)
#pragma unroll
    for (int c = 0; c < 2; ++c) k[j][c] = packed2_join(k[j][c]);
}
// s[c][h] += t_j[h] * key_j[c][h] over the digits j < beta (key words as loaded)
template <int NB>
__device__ __forceinline__ void mac_digits(double &s00, double &s01, double &s10, double &s11, const ulonglong2 (&t)[NB],
                                           const ulonglong2 (&k)[NB][2], int beta, int ext_f64, int own, const ModConst &m) {
#pragma unroll
  for (int j = 0; j < NB; ++j)
    if (j < beta) {
      // converted digits may arrive as raw lazy doubles straight from the transform (own-digit limbs are always words)
      const bool f64 = ext_f64 && j != own;
      const double t0 = f64 ? __longlong_as_double((long long)t[j].x) : u64_to_f64(t[j].x);
      const double t1 = f64 ? __longlong_as_double((long long)t[j].y) : u64_to_f64(t[j].y);
      s00 += mulmod_var(t0, u64_to_f64(k[j][0].x), m.q, m.qinv);
      s01 += mulmod_var(t1, u64_to_f64(k[j][0].y), m.q, m.qinv);
      s10 += mulmod_var(t0, u64_to_f64(k[j][1].x), m.q, m.qinv);
      s11 += mulmod_var(t1, u64_to_f64(k[j][1].y), m.q, m.qinv);
    }
}

// calls f(std::integral_constant<int, NB>()) with the digit bound NB in {1, 2, 3, 4, 8} of the kernels for beta <= 8
template <class F>
static void with_max_beta(int beta, F &&f) {
  if (beta <= 1) f(std::integral_constant<int, 1>());
  else if (beta <= 2) f(std::integral_constant<int, 2>());
  else if (beta <= 3) f(std::integral_constant<int, 3>());
  else if (beta <= 4) f(std::integral_constant<int, 4>());
  else f(std::integral_constant<int, 8>());
}

// MULTI: more than one ciphertext per launch (the next ciphertext's digits are prefetched while this one is multiplied)
// TENSOR (MULTI only, Q-limbs only): the tensor product (InnerArgs::ct_a); a1 travels as the own digit, a0, b0, b1 beside it
template <int IP_MAX_BETA, bool MULTI, bool TENSOR>
__global__ void __launch_bounds__(EW_THREADS, TENSOR ? 2 : 3) k_inner(const ModConst *__restrict__ mc, LimbMap lm, InnerArgs a) {
  pdl_wait();
  const int i2 = blockIdx.x * EW_THREADS + threadIdx.x;
  if (i2 >= a.N / 2) return;
  const int e = blockIdx.y;
  const ModConst m = mc[lm.mod[e]];
  const int kl = lm.pos[e], own = lm.skip[e];
  const size_t n2 = a.N / 2;
  constexpr bool tq = TENSOR;
  // all loads of the first ciphertext (digits + key words) are issued together; afterwards the next ciphertext's
  // digits are in flight while the current one is multiplied
  auto digit_ptr = [&](int b, int j) {
    if (tq && j == own) return a.ct_a + (size_t)b * a.ct_batch_stride + a.ct_comp_stride + (size_t)e * a.N;  // a1
    return j == own ? a.d + (size_t)b * a.d_batch_stride + (size_t)e * a.N
                    : a.ext + (size_t)b * a.ext_batch_stride + ((size_t)j * a.n_ext + e) * a.N;
  };
  ulonglong2 xn[3];  // TENSOR: a0, b0, b1 of the ciphertext the digits in flight belong to
  auto ld_tensor = [&](int b) {
    const size_t o = (size_t)b * a.ct_batch_stride + (size_t)e * a.N;
    xn[0] = ld2(a.ct_a + o, i2); xn[1] = ld2(a.ct_b + o, i2); xn[2] = ld2(a.ct_b + o + a.ct_comp_stride, i2);
  };
  if constexpr (tq) ld_tensor(0);
  const bool gal = !MULTI && a.galois != 0;  // the batched variant stays lean: no automorphism on load, no u side output
  const uint2 src = gal_slots(gal ? a.galois : 0u, a.logN, i2);
  auto ld_digit = [&](int b, int j) -> ulonglong2 {
    const u64 *p = digit_ptr(b, j);
    if (!gal) return ld2(p, i2);
    return make_ulonglong2(__ldg(p + src.x), __ldg(p + src.y));
  };
  ulonglong2 tn[IP_MAX_BETA];
#pragma unroll
  for (int j = 0; j < IP_MAX_BETA; ++j)
    if (j < a.beta) tn[j] = ld_digit(0, j);
  // every key word of the thread is requested before the first one is used: ONE memory round trip for the 3 * beta loads
  // (converting inside the load loop made ptxas wait for each digit's pair before issuing the next).  The key loads, the
  // digit loads and the product stay spelled out here: through ld_key, ld_pair or mac_digits ptxas schedules this kernel
  // differently.
  ulonglong2 kraw[IP_MAX_BETA][2];
  if (a.evk_packed) {  // uniform
#pragma unroll
    for (int j = 0; j < IP_MAX_BETA; ++j)
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        const u64 *slot = a.evk + (((size_t)j * 2 + c) * a.evk_limbs + kl) * a.N;
        kraw[j][c] = j < a.beta ? ld_packed2_raw(slot, a.N, i2) : make_ulonglong2(0, 0);
      }
    pin_loads(kraw);
    join_key(kraw);
  } else {
#pragma unroll
    for (int j = 0; j < IP_MAX_BETA; ++j)
#pragma unroll
      for (int c = 0; c < 2; ++c)
        kraw[j][c] = j < a.beta ? ld2(a.evk, (((size_t)j * 2 + c) * a.evk_limbs + kl) * n2 + i2) : make_ulonglong2(0, 0);
    pin_loads(kraw);
  }
  double k[IP_MAX_BETA][2][2];  // [digit][component][coefficient]
#pragma unroll
  for (int j = 0; j < IP_MAX_BETA; ++j)
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      k[j][c][0] = u64_to_f64(kraw[j][c].x); k[j][c][1] = u64_to_f64(kraw[j][c].y);
    }
  const double2 pm = tq ? a.tensor_pmod[e] : make_double2(0.0, 0.0);  // P mod q_e
  for (int b = 0; b < a.n_batch; ++b) {
    u64 *acc = a.acc + (size_t)b * a.acc_batch_stride;
    ulonglong2 t[IP_MAX_BETA];
#pragma unroll
    for (int j = 0; j < IP_MAX_BETA; ++j) t[j] = tn[j];
    double s00 = 0, s01 = 0, s10 = 0, s11 = 0;  // [component][coefficient]
    double o0 = 0, o1 = 0;                      // TENSOR: the own-digit term d2 = a1 * b1
    if constexpr (tq) {  // d2, and the accumulators start at d0 * P, d1 * P (before the next loads: xn is refilled below)
      ulonglong2 a1 = t[0];
#pragma unroll
      for (int j = 1; j < IP_MAX_BETA; ++j)
        if (j == own) a1 = t[j];
      const double a0x = u64_to_f64(xn[0].x), a0y = u64_to_f64(xn[0].y), a1x = u64_to_f64(a1.x), a1y = u64_to_f64(a1.y);
      const double b0x = u64_to_f64(xn[1].x), b0y = u64_to_f64(xn[1].y), b1x = u64_to_f64(xn[2].x), b1y = u64_to_f64(xn[2].y);
      o0 = mulmod_var(a1x, b1x, m.q, m.qinv);
      o1 = mulmod_var(a1y, b1y, m.q, m.qinv);
      s00 = mulmod_const(mulmod_var(a0x, b0x, m.q, m.qinv), pm.x, pm.y, m.q);
      s01 = mulmod_const(mulmod_var(a0y, b0y, m.q, m.qinv), pm.x, pm.y, m.q);
      s10 = mulmod_const(mulmod_var(a0x, b1x, m.q, m.qinv) + mulmod_var(a1x, b0x, m.q, m.qinv), pm.x, pm.y, m.q);
      s11 = mulmod_const(mulmod_var(a0y, b1y, m.q, m.qinv) + mulmod_var(a1y, b0y, m.q, m.qinv), pm.x, pm.y, m.q);
    }
    if (MULTI && b + 1 < a.n_batch) {
#pragma unroll
      for (int j = 0; j < IP_MAX_BETA; ++j)
        if (j < a.beta) tn[j] = ld_digit(b + 1, j);
      if constexpr (tq) ld_tensor(b + 1);
    }
#pragma unroll
    for (int j = 0; j < IP_MAX_BETA; ++j)
      if (j < a.beta) {
        const bool f64 = a.ext_f64 && j != own, sq = tq && j == own;
        const double t0 = sq ? o0 : f64 ? __longlong_as_double((long long)t[j].x) : u64_to_f64(t[j].x);
        const double t1 = sq ? o1 : f64 ? __longlong_as_double((long long)t[j].y) : u64_to_f64(t[j].y);
        s00 += mulmod_var(t0, k[j][0][0], m.q, m.qinv);
        s01 += mulmod_var(t1, k[j][0][1], m.q, m.qinv);
        s10 += mulmod_var(t0, k[j][1][0], m.q, m.qinv);
        s11 += mulmod_var(t1, k[j][1][1], m.q, m.qinv);
      }
    const size_t comp2 = (a.acc_comp_stride ? (size_t)a.acc_comp_stride : (size_t)a.n_ext * a.N) / 2;
    const u64 r00 = finish(s00, m), r01 = finish(s01, m), r10 = finish(s10, m), r11 = finish(s11, m);
    if (e < a.acc_pack_limbs) {  // uniform per CTA
      st_packed2(acc + (size_t)e * a.N, a.N, i2, r00, r01);
      st_packed2(acc + 2 * comp2 + (size_t)e * a.N, a.N, i2, r10, r11);
    } else {
      st2(acc, (size_t)e * n2 + i2, r00, r01);
      st2(acc, comp2 + (size_t)e * n2 + i2, r10, r11);
    }
    if (!MULTI && e == a.u_limb) {  // uniform per CTA: u = acc * P^-1 + d on the limb the rescale drops (no extra launch, no re-read)
      const u64 *ua = a.u_add + (size_t)b * a.u_add_batch_stride + (size_t)e * a.N;
      const ulonglong2 d0v = ld_packed2(ua, a.N, i2), d1v = ld_packed2(ua + a.u_add_comp_stride, a.N, i2);
      const double2 c = a.u_cst;
      st2(acc, (size_t)a.u_slot * n2 + i2, finish(mulmod_const(u64_to_f64(r00), c.x, c.y, m.q) + u64_to_f64(d0v.x), m),
          finish(mulmod_const(u64_to_f64(r01), c.x, c.y, m.q) + u64_to_f64(d0v.y), m));
      st2(acc, comp2 + (size_t)a.u_slot * n2 + i2, finish(mulmod_const(u64_to_f64(r10), c.x, c.y, m.q) + u64_to_f64(d1v.x), m),
          finish(mulmod_const(u64_to_f64(r11), c.x, c.y, m.q) + u64_to_f64(d1v.y), m));
    }
  }
}

void launch_inner_product(const ModConst *mc, const LimbMap &lm, const InnerArgs &a, cudaStream_t s, int n_limbs) {
  const dim3 grid = ew_grid(a.N, n_limbs ? n_limbs : a.n_ext);
  with_max_beta(a.beta, [&](auto nb) {
    constexpr int NB = decltype(nb)::value;
    if (a.n_batch > 1 && a.ct_a) launch_pdl(k_inner<NB, true, true>, grid, EW_THREADS, 0, s, mc, lm, a);
    else if (a.n_batch > 1) launch_pdl(k_inner<NB, true, false>, grid, EW_THREADS, 0, s, mc, lm, a);
    else launch_pdl(k_inner<NB, false, false>, grid, EW_THREADS, 0, s, mc, lm, a);
  });
}

// Hoisted rotations of one ciphertext (limb-sharded, shard.cu): k_inner's single-ciphertext body with the automorphism on
// load, once per rotation (blockIdx.z), each with its own key and galois element.  Rotations are the slowest grid dimension,
// so the digits stay in L2 while the later rotations re-read them.  Five to eight digits need 128 registers (two CTAs per SM)
// to hold the 32 key words without spilling.
template <int IP_MAX_BETA>
__global__ void __launch_bounds__(EW_THREADS, IP_MAX_BETA > 4 ? 2 : 3) k_inner_rot(const ModConst *__restrict__ mc, LimbMap lm, InnerRotArgs a) {
  pdl_wait();
  const int i2 = blockIdx.x * EW_THREADS + threadIdx.x;
  if (i2 >= a.N / 2) return;
  const int e = blockIdx.y, r = blockIdx.z;
  const ModConst m = mc[lm.mod[e]];
  const int kl = lm.pos[e], own = lm.skip[e];
  const size_t n2 = a.N / 2;
  const unsigned g = a.galois[r];
  const u64 *evk = a.evk[r];
  const uint2 src = gal_slots(g, a.logN, i2);
  ulonglong2 t[IP_MAX_BETA];
#pragma unroll
  for (int j = 0; j < IP_MAX_BETA; ++j)
    if (j < a.beta) {
      const u64 *p = j == own ? a.d + (size_t)e * a.N : a.ext + ((size_t)j * a.n_ext + e) * a.N;
      t[j] = ld_pair(p, i2, src, g != 0);
    }
  ulonglong2 kraw[IP_MAX_BETA][2];  // every key word requested before the first use
  ld_key<false>(kraw, evk, a, kl, n2, i2);
  pin_loads(kraw);
  double s00 = 0, s01 = 0, s10 = 0, s11 = 0;  // [component][coefficient]
  mac_digits(s00, s01, s10, s11, t, kraw, a.beta, a.ext_f64, own, m);
  u64 *acc = a.acc + (size_t)r * a.acc_rot_stride;
  st2(acc, (size_t)e * n2 + i2, finish(s00, m), finish(s01, m));
  st2(acc, (size_t)(a.n_ext + e) * n2 + i2, finish(s10, m), finish(s11, m));
}

void launch_inner_product_rot(const ModConst *mc, const LimbMap &lm, const InnerRotArgs &a, int n_rot, cudaStream_t s) {
  with_max_beta(a.beta, [&](auto nb) {
    launch_pdl(k_inner_rot<decltype(nb)::value>, ew_grid(a.N, a.n_ext, n_rot), EW_THREADS, 0, s, mc, lm, a);
  });
}

// Double-hoisted rotation sum (ewe.cuh InnerRotSumArgs).  The body of k_inner_rot once per rotation, then the two component
// sums are weighted by the plaintext and kept in registers: the op is bound by reading the keys, and every rotation's key,
// plaintext and c0 loads are issued before its first use.  The argument table is read in place (grid constant), so the
// rotation index may be a loop variable.  Exact: |sum_j| <= 8 * 0.51 q, each weighted term <= 0.51 q, 16 terms + one stored
// word stay far below 2^51.  PACKED (the key's load path) is a template argument: with both paths in one body four digits
// spilled at 128 registers.  Up to three digits fit three CTAs per SM (76 registers), four digits two (108-128), five to eight
// digits one (229-237).
// MODE selects the kernel the body serves: RS_SUM k_inner_rot_sum; RS_BABY and RS_GIANT k_inner_bsgs (ewe.cuh InnerBsgsArgs).
enum { RS_SUM, RS_BABY, RS_GIANT };
template <int IP_MAX_BETA, bool PACKED, int MODE, class A>
__device__ __forceinline__ void rot_sum_body(const ModConst *__restrict__ mc, const LimbMap &lm, const A &a, int i2) {
  const int e = blockIdx.y;
  const ModConst m = mc[lm.mod[e]];
  const int kl = lm.pos[e], own = lm.skip[e];
  const size_t n2 = a.N / 2;
  const bool q_limb = e < a.L;  // uniform per CTA
  const size_t prow = q_limb ? (size_t)e : (size_t)a.pt_q_limbs + (e - a.L);
  double a00 = 0, a01 = 0, a10 = 0, a11 = 0, z0 = 0, z1 = 0;  // [component][coefficient], z = the c0 term
  double y0 = 0, y1 = 0;                                       // RS_BABY: the c1 term of the identity entries
#pragma unroll 1
  for (int r = 0; r < a.n_rot; ++r) {
    if constexpr (MODE == RS_BABY) {
      if (!a.evk[r]) {  // uniform: the identity without a key switch, nothing on the P-limbs
        if (q_limb) {
          const ulonglong2 w = ld2(a.pt[r] + prow * a.N, i2), x = ld2(a.c0 + (size_t)e * a.N, i2), y = ld2(a.d + (size_t)e * a.N, i2);
          const double w0 = u64_to_f64(w.x), w1 = u64_to_f64(w.y);
          z0 += mulmod_var(u64_to_f64(x.x), w0, m.q, m.qinv);
          z1 += mulmod_var(u64_to_f64(x.y), w1, m.q, m.qinv);
          y0 += mulmod_var(u64_to_f64(y.x), w0, m.q, m.qinv);
          y1 += mulmod_var(u64_to_f64(y.y), w1, m.q, m.qinv);
        }
        continue;
      }
    }
    const unsigned g = a.galois[r];
    const uint2 src = gal_slots(g, a.logN, i2);
    ulonglong2 t[IP_MAX_BETA];
#pragma unroll
    for (int j = 0; j < IP_MAX_BETA; ++j)
      if (j < a.beta) {
        const u64 *p = j == own ? a.d + (size_t)e * a.N : a.ext + ((size_t)j * a.n_ext + e) * a.N;
        t[j] = ld_pair(p, i2, src, g != 0);
      }
    ulonglong2 kraw[IP_MAX_BETA][2];
    ld_key<PACKED>(kraw, a.evk[r], a, kl, n2, i2);
    ulonglong2 w = make_ulonglong2(0, 0), x = make_ulonglong2(0, 0);
    if constexpr (MODE != RS_GIANT) w = ld2(a.pt[r] + prow * a.N, i2);
    if (q_limb) x = ld_pair(a.c0 + (size_t)e * a.N, i2, src, g != 0);
    pin_loads(kraw);
    if constexpr (MODE != RS_GIANT) asm volatile("" : "+l"(w.x), "+l"(w.y), "+l"(x.x), "+l"(x.y));
    else asm volatile("" : "+l"(x.x), "+l"(x.y));
    if constexpr (PACKED) join_key(kraw);
    double s00 = 0, s01 = 0, s10 = 0, s11 = 0;
    mac_digits(s00, s01, s10, s11, t, kraw, a.beta, a.ext_f64, own, m);
    if constexpr (MODE == RS_GIANT) {  // unweighted: one term of at most 8 * 0.51 q per rotation
      a00 += s00; a01 += s01; a10 += s10; a11 += s11;
      if (q_limb) { z0 += u64_to_f64(x.x); z1 += u64_to_f64(x.y); }
    } else {
      const double w0 = u64_to_f64(w.x), w1 = u64_to_f64(w.y);
      a00 += mulmod_var(s00, w0, m.q, m.qinv);
      a01 += mulmod_var(s01, w1, m.q, m.qinv);
      a10 += mulmod_var(s10, w0, m.q, m.qinv);
      a11 += mulmod_var(s11, w1, m.q, m.qinv);
      if (q_limb) {
        z0 += mulmod_var(u64_to_f64(x.x), w0, m.q, m.qinv);
        z1 += mulmod_var(u64_to_f64(x.y), w1, m.q, m.qinv);
      }
    }
  }
  const size_t o0 = (size_t)e * n2 + i2, o1 = (size_t)(a.n_ext + e) * n2 + i2;
  if (a.accumulate) {  // uniform: a later group of the same op
    const ulonglong2 p0 = ld2(a.acc, o0), p1 = ld2(a.acc, o1);
    a00 += u64_to_f64(p0.x); a01 += u64_to_f64(p0.y); a10 += u64_to_f64(p1.x); a11 += u64_to_f64(p1.y);
    if (q_limb) {
      const ulonglong2 pz = ld2(a.z, o0);
      z0 += u64_to_f64(pz.x); z1 += u64_to_f64(pz.y);
      if constexpr (MODE == RS_BABY) {
        const ulonglong2 py = ld2(a.z1, o0);
        y0 += u64_to_f64(py.x); y1 += u64_to_f64(py.y);
      }
    }
  }
  st2(a.acc, o0, finish(a00, m), finish(a01, m));
  st2(a.acc, o1, finish(a10, m), finish(a11, m));
  if (q_limb) st2(a.z, o0, finish(z0, m), finish(z1, m));
  if constexpr (MODE == RS_BABY)
    if (q_limb) st2(a.z1, o0, finish(y0, m), finish(y1, m));
}

template <int IP_MAX_BETA, bool PACKED>
__global__ void __launch_bounds__(EW_THREADS, IP_MAX_BETA > 4 ? 1 : IP_MAX_BETA > 3 ? 2 : 3)
    k_inner_rot_sum(const ModConst *__restrict__ mc, LimbMap lm, const __grid_constant__ InnerRotSumArgs a) {
  pdl_wait();
  const int i2 = blockIdx.x * EW_THREADS + threadIdx.x;
  if (i2 >= a.N / 2) return;
  rot_sum_body<IP_MAX_BETA, PACKED, RS_SUM>(mc, lm, a, i2);
}

void launch_inner_product_rot_sum(const ModConst *mc, const LimbMap &lm, const InnerRotSumArgs &a, cudaStream_t s) {
  with_max_beta(a.beta, [&](auto nb) {
    constexpr int NB = decltype(nb)::value;
    if (a.evk_packed) launch_pdl(k_inner_rot_sum<NB, true>, ew_grid(a.N, a.n_ext), EW_THREADS, 0, s, mc, lm, a);
    else launch_pdl(k_inner_rot_sum<NB, false>, ew_grid(a.N, a.n_ext), EW_THREADS, 0, s, mc, lm, a);
  });
}

// The two inner products of a double-hoisted BSGS linear transform (ewe.cuh InnerBsgsArgs), k_inner_rot_sum's body with
// identity entries (GIANT = false) or without the plaintext (GIANT = true)
template <int IP_MAX_BETA, bool PACKED, bool GIANT>
__global__ void __launch_bounds__(EW_THREADS, IP_MAX_BETA > 4 ? 1 : IP_MAX_BETA > 3 ? 2 : 3)
    k_inner_bsgs(const ModConst *__restrict__ mc, LimbMap lm, const __grid_constant__ InnerBsgsArgs a) {
  pdl_wait();
  const int i2 = blockIdx.x * EW_THREADS + threadIdx.x;
  if (i2 >= a.N / 2) return;
  rot_sum_body<IP_MAX_BETA, PACKED, GIANT ? RS_GIANT : RS_BABY>(mc, lm, a, i2);
}

void launch_inner_product_bsgs(const ModConst *mc, const LimbMap &lm, const InnerBsgsArgs &a, bool giant, cudaStream_t s) {
  with_max_beta(a.beta, [&](auto nb) {
    constexpr int NB = decltype(nb)::value;
    const dim3 grid = ew_grid(a.N, a.n_ext);
    if (giant) {
      if (a.evk_packed) launch_pdl(k_inner_bsgs<NB, true, true>, grid, EW_THREADS, 0, s, mc, lm, a);
      else launch_pdl(k_inner_bsgs<NB, false, true>, grid, EW_THREADS, 0, s, mc, lm, a);
    } else {
      if (a.evk_packed) launch_pdl(k_inner_bsgs<NB, true, false>, grid, EW_THREADS, 0, s, mc, lm, a);
      else launch_pdl(k_inner_bsgs<NB, false, false>, grid, EW_THREADS, 0, s, mc, lm, a);
    }
  });
}

// ------------------------------------------------------------------------------------------------ (x - y) * c (+ z)
__global__ void __launch_bounds__(EW_THREADS) k_sub_mul_add(const ModConst *__restrict__ mc, LimbMap lm, SubMulArgs a) {
  pdl_wait();
  const int i2 = blockIdx.x * EW_THREADS + threadIdx.x;
  if (i2 >= a.N / 2) return;
  const int limb = blockIdx.y, poly = blockIdx.z;
  const ModConst m = mc[lm.mod[limb]];
  const double2 c = a.cst[limb];
  const size_t o = (size_t)limb * (a.N / 2) + i2;
  const ulonglong2 x = a.x_packed ? ld_packed2(a.x + poly * a.x_poly_stride + (size_t)limb * a.N, a.N, i2) : ld2(a.x + poly * a.x_poly_stride, o);
  const ulonglong2 y = a.y ? ld2(a.y + poly * a.y_poly_stride, o) : make_ulonglong2(0, 0);
  double r0 = mulmod_const(u64_to_f64(x.x) - u64_to_f64(y.x), c.x, c.y, m.q);
  double r1 = mulmod_const(u64_to_f64(x.y) - u64_to_f64(y.y), c.x, c.y, m.q);
  if (a.z && (a.z_mask == 0 || ((a.z_mask >> poly) & 1u))) {
    const ulonglong2 z = a.z_packed ? ld_packed2(a.z + poly * a.z_poly_stride + (size_t)limb * a.N, a.N, i2) : ld2(a.z + poly * a.z_poly_stride, o);
    r0 += u64_to_f64(z.x);
    r1 += u64_to_f64(z.y);
  }
  st2(a.out + poly * a.out_poly_stride, o, finish(r0, m), finish(r1, m));
}

void launch_sub_mul_add(const ModConst *mc, const LimbMap &lm, const SubMulArgs &a, cudaStream_t s) {
  launch_pdl(k_sub_mul_add, ew_grid(a.N, a.n_limbs, a.n_polys), EW_THREADS, 0, s, mc, lm, a);
}

// ------------------------------------------------------------------------------------------------ automorphism
__global__ void __launch_bounds__(EW_THREADS) k_automorph(int logN, const u64 *__restrict__ in, u64 *__restrict__ out, unsigned g) {
  pdl_wait();
  const unsigned N = 1u << logN;
  const unsigned k = blockIdx.x * EW_THREADS + threadIdx.x;
  if (k >= N) return;
  const unsigned j = __brev(k) >> (32 - logN);
  const unsigned e = (g * (2u * j + 1u)) & (2u * N - 1u);  // low bits of the product are exact
  const unsigned ks = __brev((e - 1u) >> 1) >> (32 - logN);
  const size_t base = (size_t)blockIdx.y << logN;
  out[base + k] = __ldg(&in[base + ks]);
}

void launch_automorph(int logN, int n_limbs, const u64 *in, u64 *out, u64 g, cudaStream_t s) {
  const unsigned N = 1u << logN;
  launch_pdl(k_automorph, dim3((N + EW_THREADS - 1) / EW_THREADS, n_limbs), EW_THREADS, 0, s, logN, in, out, (unsigned)(g & (2ull * N - 1)));
}

// words -> packed limbs, slot geometry unchanged (evaluation keys: hml_key_pack)
__global__ void __launch_bounds__(EW_THREADS) k_pack_limbs(int N, const u64 *__restrict__ in, u64 *__restrict__ out) {
  pdl_wait();
  const size_t i2 = (size_t)blockIdx.x * EW_THREADS + threadIdx.x;
  if (i2 >= (size_t)N / 2) return;
  const size_t limb = blockIdx.y + (size_t)blockIdx.z * gridDim.y;
  const ulonglong2 v = ld2(in + limb * N, i2);
  st_packed2(out + limb * N, N, i2, v.x, v.y);
}
void launch_pack_limbs(int N, size_t n_limbs, const u64 *in, u64 *out, cudaStream_t s) {
  for (size_t done = 0; done < n_limbs;) {  // grid.y * grid.z limbs per launch
    const size_t rest = n_limbs - done, gy = rest < 256 ? rest : 256, gz = std::min<size_t>(rest / gy, 65535);
    launch_pdl(k_pack_limbs, dim3((unsigned)((N / 2 + EW_THREADS - 1) / EW_THREADS), (unsigned)gy, (unsigned)gz), EW_THREADS, 0, s, N, in + done * N, out + done * N);
    done += gy * gz;
  }
}

// ------------------------------------------------------------------------------------------------ base conversion
// out[t][m] = sum_i y_i[m] * H[i][t]  (mod q_t)  is a matrix product [coefficients x sources] x [sources x targets]
// with exact integer entries.  It runs on the FP64 tensor-core path (DMMA m8n8k4): H is split into three 12-bit pieces
// so that every product (36 + 12 bits) and every 16-term partial sum (<= 52 bits) is an exactly representable double,
// whatever the accumulation order inside the MMA.  Measured on B200 (profiles/microbench/dmma_bench.cu): DMMA reaches
// the FP64 pipe's full 18.5 T FMA/s with ONE instruction per 256 FMAs, and integer / load instructions issue in its
// shadow, whereas a DFMA holds the issue port for two cycles per 32 FMAs — the earlier DFMA kernel spent 25% of its
// issue slots on matrix-operand loads alone.
//   CTA  = `tm` coefficients (256, or 64 when there are many sources) x all targets; the sources of the tile are
//          staged once in shared memory as doubles, pitch tm + 4 (conflict-free fragment reads), zero rows as padding
//   warp = one block of 8 targets: B fragments (sources x 8 targets x 3 pieces) live in registers for <= 16 sources
//          (KS = number of 4-source k-steps), else they are re-read from the L1-resident matrix and the accumulators are
//          folded mod q_t every 16 sources
//   lane = coefficient lane/4 of each 8-coefficient m-tile, targets 2*(lane%4), +1 of the block: the three pieces of a
//          target meet in one lane, so the epilogue (Horner over the pieces, 3 reductions) needs no exchange
__device__ __forceinline__ void dmma884(double &d0, double &d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

template <int KS, bool STEP1>
__global__ void __launch_bounds__(512) k_bconv_mma(const ModConst *__restrict__ mc, LimbMap src_lm, LimbMap dst_lm, BConvArgs a,
                                                   const double *__restrict__ mat, int n_src_pad, int n_dst_pad, int tm) {
  extern __shared__ __align__(16) double ys[];  // [n_src_pad][tm + 4]
  const int pitch = tm + 4;
  const int lane = threadIdx.x & 31, tb = threadIdx.x >> 5;
  const size_t m_base = (size_t)blockIdx.x * tm;
  const u64 *in = a.in + (size_t)blockIdx.y * a.in_batch_stride;
  u64 *out = a.out + (size_t)blockIdx.y * a.out_batch_stride;
  // matrix fragments and moduli are constant tables: fetched before the programmatic dependency is resolved
  const bool mma_warp = tb * 8 < n_dst_pad;  // a launch with fewer than four target blocks has staging-only helper warps
  const int kq = lane & 3, rq = lane >> 2;
  const int t0 = tb * 8 + 2 * kq, t1 = t0 + 1;
  const bool live0 = t0 < a.n_dst, live1 = t1 < a.n_dst;
  const ModConst m0 = mc[dst_lm.mod[live0 ? t0 : a.n_dst - 1]], m1 = mc[dst_lm.mod[live1 ? t1 : a.n_dst - 1]];
  u64 *o0 = out + (size_t)dst_lm.pos[live0 ? t0 : a.n_dst - 1] * a.N + m_base + rq;
  u64 *o1 = out + (size_t)dst_lm.pos[live1 ? t1 : a.n_dst - 1] * a.N + m_base + rq;
  const double *bsrc = mat + ((size_t)kq * n_dst_pad + tb * 8 + rq) * 3;  // B[k = lane%4][n = lane/4], k-step stride 4 rows
  const size_t brow = (size_t)4 * n_dst_pad * 3;
  double bf[KS > 0 ? KS : 1][3];
  if constexpr (KS > 0) {
#pragma unroll
    for (int ks = 0; ks < KS; ++ks)
#pragma unroll
      for (int p = 0; p < 3; ++p) bf[ks][p] = mma_warp ? __ldg(bsrc + ks * brow + p) : 0.0;
  }
  pdl_wait();  // the sources are another kernel's output
  {  // stage the tile's sources (step 1 applied here when requested), zero the padding rows; four loads in flight per thread
    const int half = tm >> 1, total = n_src_pad * half;
    for (int e0 = threadIdx.x; e0 < total; e0 += 4 * blockDim.x) {
      ulonglong2 v[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int e = e0 + k * blockDim.x, i = e / half, m2 = e - i * half;
        v[k] = make_ulonglong2(0, 0);
        if (e < total && i < a.n_src) v[k] = __ldg(reinterpret_cast<const ulonglong2 *>(in + (size_t)src_lm.pos[i] * a.N + m_base) + m2);
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int e = e0 + k * blockDim.x, i = e / half, m2 = e - i * half;
        if (e >= total) break;
        double y0 = u64_to_f64(v[k].x), y1 = u64_to_f64(v[k].y);
        if (STEP1 && i < a.n_src) {
          const ModConst m = mc[src_lm.mod[i]];
          const double2 sc = a.step1[i];
          y0 = canonicalize(mulmod_const(y0, sc.x, sc.y, m.q), m.q);
          y1 = canonicalize(mulmod_const(y1, sc.x, sc.y, m.q), m.q);
        }
        *reinterpret_cast<double2 *>(&ys[i * pitch + 2 * m2]) = make_double2(y0, y1);
      }
    }
  }
  __syncthreads();
  if (a.fold) {  // uniform branch: every thread of the CTA takes it
    const ModConst mf = mc[a.fold_mod];
    const int last = a.n_src - 1;
    for (int m = threadIdx.x; m < tm; m += blockDim.x) {
      double s0 = 0.0, s1 = 0.0, s2 = 0.0;  // terms of < 2^48 each: exact as long as at most 16 are summed unreduced
      for (int i = 0; i < last; ++i) {
        const double y = ys[i * pitch + m];
        s0 = __fma_rn(y, __ldg(a.fold + 3 * i), s0);
        s1 = __fma_rn(y, __ldg(a.fold + 3 * i + 1), s1);
        s2 = __fma_rn(y, __ldg(a.fold + 3 * i + 2), s2);
        if ((i & 15) == 15) {  // alpha > 16 (DMMA path only): fold like the main loop does, every 16 sources
          s0 = reduce_signed(s0, mf.q, mf.qinv);
          s1 = reduce_signed(s1, mf.q, mf.qinv);
          s2 = reduce_signed(s2, mf.q, mf.qinv);
        }
      }
      double v = reduce_signed(s2, mf.q, mf.qinv);
      v = reduce_signed(__fma_rn(v, 4096.0, s1), mf.q, mf.qinv);
      v = reduce_signed(__fma_rn(v, 4096.0, s0 + ys[last * pitch + m]), mf.q, mf.qinv);
      ys[last * pitch + m] = canonicalize(v, mf.q);
    }
    __syncthreads();
  }
  if (!mma_warp) return;
  const double nh0 = a.out_f64 ? 0.0 : -(m0.q - 1.0) * 0.5, nh1 = a.out_f64 ? 0.0 : -(m1.q - 1.0) * 0.5;
  const double hb0 = 4503599627370496.0 - nh0, hb1 = 4503599627370496.0 - nh1;  // 2^52 + h
  const double *yl = ys + kq * pitch + rq;  // A[row = lane/4][col = lane%4]
  const int n_ks = n_src_pad >> 2;
  // two m-tiles (16 coefficients) per iteration: six independent accumulator chains keep the tensor pipe fed
  for (int mt = 0; mt < (tm >> 3); mt += 2) {
    // piece-0 accumulators start at -h, h = (q_t - 1) / 2: the final centred remainder is then (value - h) in [-h, h] and
    // canonicalisation is one add of 2^52 + h (no sign fix-up)
    double acc[2][3][2] = {{{nh0, nh1}, {0.0, 0.0}, {0.0, 0.0}}, {{nh0, nh1}, {0.0, 0.0}, {0.0, 0.0}}};
    if constexpr (KS > 0) {
#pragma unroll
      for (int ks = 0; ks < KS; ++ks) {
        const double af0 = yl[ks * 4 * pitch + mt * 8], af1 = yl[ks * 4 * pitch + mt * 8 + 8];
#pragma unroll
        for (int p = 0; p < 3; ++p) {
          dmma884(acc[0][p][0], acc[0][p][1], af0, bf[ks][p]);
          dmma884(acc[1][p][0], acc[1][p][1], af1, bf[ks][p]);
        }
      }
    } else {
      for (int ks = 0; ks < n_ks; ++ks) {
        const double af0 = yl[ks * 4 * pitch + mt * 8], af1 = yl[ks * 4 * pitch + mt * 8 + 8];
#pragma unroll
        for (int p = 0; p < 3; ++p) {
          const double b = __ldg(bsrc + ks * brow + p);
          dmma884(acc[0][p][0], acc[0][p][1], af0, b);
          dmma884(acc[1][p][0], acc[1][p][1], af1, b);
        }
        // each term is < 2^36 * 2^12: fold every 16 sources so the exact sums stay below 2^53
        if ((ks & 3) == 3 && ks + 1 < n_ks) {
#pragma unroll
          for (int h = 0; h < 2; ++h)
#pragma unroll
            for (int p = 0; p < 3; ++p) {
              acc[h][p][0] = reduce_signed(acc[h][p][0], m0.q, m0.qinv);
              acc[h][p][1] = reduce_signed(acc[h][p][1], m1.q, m1.qinv);
            }
        }
      }
    }
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      // value = S2*2^24 + S1*2^12 + S0 (mod q), folded top-down; every intermediate is an exact integer < 2^53
      double v0 = reduce_signed(acc[h][2][0], m0.q, m0.qinv), v1 = reduce_signed(acc[h][2][1], m1.q, m1.qinv);
      v0 = reduce_signed(__fma_rn(v0, 4096.0, acc[h][1][0]), m0.q, m0.qinv);
      v1 = reduce_signed(__fma_rn(v1, 4096.0, acc[h][1][1]), m1.q, m1.qinv);
      v0 = reduce_signed(__fma_rn(v0, 4096.0, acc[h][0][0]), m0.q, m0.qinv);
      v1 = reduce_signed(__fma_rn(v1, 4096.0, acc[h][0][1]), m1.q, m1.qinv);
      if (a.out_f64) {  // uniform
        if (live0) reinterpret_cast<double *>(o0)[(mt + h) * 8] = v0;
        if (live1) reinterpret_cast<double *>(o1)[(mt + h) * 8] = v1;
      } else {
        if (live0) o0[(mt + h) * 8] = (u64)__double_as_longlong(v0 + hb0) & 0x000FFFFFFFFFFFFFull;
        if (live1) o1[(mt + h) * 8] = (u64)__double_as_longlong(v1 + hb1) & 0x000FFFFFFFFFFFFFull;
      }
    }
  }
}

template <int KS>
static void launch_bconv_t(const ModConst *mc, const LimbMap &src_lm, const LimbMap &dst_lm, const BConvArgs &a, const double *mat,
                           int n_src_pad, int n_dst_pad, int tm, cudaStream_t s) {
  const dim3 grid(a.N / tm, a.n_batches);
  const int threads = std::max(128, 32 * (n_dst_pad / 8));  // at least four warps so that staging has loads in flight
  const size_t smem = (size_t)n_src_pad * (tm + 4) * sizeof(double);
  static PerDeviceOnce once;
  if (once.first()) {
    cudaFuncSetAttribute(k_bconv_mma<KS, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 68 * 8);
    cudaFuncSetAttribute(k_bconv_mma<KS, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 68 * 8);
  }
  if (a.step1) launch_pdl(k_bconv_mma<KS, true>, grid, threads, smem, s, mc, src_lm, dst_lm, a, mat, n_src_pad, n_dst_pad, tm);
  else launch_pdl(k_bconv_mma<KS, false>, grid, threads, smem, s, mc, src_lm, dst_lm, a, mat, n_src_pad, n_dst_pad, tm);
}

int bconv_umma_enabled() {
  static const int v = [] {
    const char *e = getenv("HML_BCONV_UMMA");
    return e && atoi(e) == 0 ? 0 : 1;
  }();
  return v;
}

void launch_bconv(const ModConst *mc, const LimbMap &src_lm, const LimbMap &dst_lm, const BConvArgs &a, const double *mat, cudaStream_t s,
                  const BConvImage *im) {
  if (im && im->img && a.N >= 128 && a.N % 128 == 0 && (a.fold != nullptr) == (im->fold != 0) && bconv_umma_enabled()) {
    launch_bconv_umma(mc, src_lm, dst_lm, a, *im, s);
    return;
  }
  const int n_src_pad = bconv_pad_src(a.n_src), n_dst_pad = bconv_pad_dst(a.n_dst);
  // big tiles amortise the per-CTA set-up (matrix fragments, moduli); small launches need more, shorter CTAs to fill 148 SMs
  int tm = 64;
  if (n_src_pad <= 16) {
    tm = 256;
    while (tm > 64 && (long long)(a.N / tm) * a.n_batches < 1480) tm >>= 1;
  }
  while (tm > a.N) tm >>= 1;  // tiny rings (tests): N >= 16
  switch (n_src_pad <= 16 ? n_src_pad / 4 : 0) {
    case 1: launch_bconv_t<1>(mc, src_lm, dst_lm, a, mat, n_src_pad, n_dst_pad, tm, s); break;
    case 2: launch_bconv_t<2>(mc, src_lm, dst_lm, a, mat, n_src_pad, n_dst_pad, tm, s); break;
    case 3: launch_bconv_t<3>(mc, src_lm, dst_lm, a, mat, n_src_pad, n_dst_pad, tm, s); break;
    case 4: launch_bconv_t<4>(mc, src_lm, dst_lm, a, mat, n_src_pad, n_dst_pad, tm, s); break;
    default: launch_bconv_t<0>(mc, src_lm, dst_lm, a, mat, n_src_pad, n_dst_pad, tm, s); break;
  }
}

}  // namespace hml
