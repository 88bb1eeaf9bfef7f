// Device-side modular arithmetic for word sizes <= 36 bits, carried out on B200's FP64 pipe.
//
// Why FP64: measured on B200 (profiles/microbench/butterfly_bench.cu, profiles/microbench_r1.txt)
//   IMAD.WIDE.U32 / IMAD.HI.U32   32 lane-ops/clk/SM      IMAD (32-bit)   64
//   IADD3 / LOP3                 128                      DFMA            64
// A 64-bit Shoup butterfly needs ~10 wide IMADs (870 G butterflies/s measured); the same butterfly on
// doubles holding exact integers needs 8 DP ops (2027 G butterflies/s measured, 2.3x).  B200 (sm_100a)
// keeps the full-rate FP64 pipe (B300 does not), so this is a B200-specific choice.
//
// Representation: a residue is a double holding an exact integer, either canonical [0,q) or "signed
// lazy" with |v| < 2^51.  Every operation below is EXACT (no rounding ever reaches a result):
//   * products a*b are split error-free: h = RN(a*b), l = fma(a,b,-h)  (l is always representable)
//   * the quotient estimate qh = rint(a*b/q) is off by at most +-1/2 + 2^-9, so the remainder
//     r = fma(-qh, q, h) + l is an integer of magnitude < 0.51*q + 2^25 < 2^53: exact.
// Requirements, enforced at context creation: q < 2^36, and the caller keeps |inputs| < 2^44.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace hml {

typedef unsigned long long u64;

// 1.5 * 2^52: adding it to x (|x| < 2^51) rounds x to the nearest integer in the low mantissa bits
#define HML_MAGIC 6755399441055744.0

// ---- integer <-> double (exact for 0 <= x < 2^52)
__device__ __forceinline__ double u64_to_f64(u64 x) {
  // (2^52 | x) reinterpreted is exactly 2^52 + x
  return __longlong_as_double((long long)(x | 0x4330000000000000ull)) - 4503599627370496.0;
}
// signed lazy value (|v| < 2^51, integer) -> canonical [0,q) as u64.  v must already satisfy |v| < q.
__device__ __forceinline__ u64 f64_to_canonical(double v, u64 q) {
  long long s = __double_as_longlong(v + HML_MAGIC) - 0x4338000000000000ll;  // exact signed integer
  return (u64)(s + ((s >> 63) & (long long)q));
}
__device__ __forceinline__ double canonicalize(double v, double q) { return v < 0.0 ? v + q : v; }

// ---- v mod q, result in [-q/2 - eps, q/2 + eps]  (|v| < 2^51)
__device__ __forceinline__ double reduce_signed(double v, double q, double qinv) {
  double qh = __fma_rn(v, qinv, HML_MAGIC) - HML_MAGIC;
  return __fma_rn(-qh, q, v);
}

// ---- a*w mod q with a precomputed wq = RN(w/q) (Shoup-style constant multiplier); signed result, |r| <= 0.51 q
__device__ __forceinline__ double mulmod_const(double a, double w, double wq, double q) {
  double qh = __fma_rn(a, wq, HML_MAGIC) - HML_MAGIC;
  double h = __dmul_rn(a, w);
  double l = __fma_rn(a, w, -h);
  double r = __fma_rn(-qh, q, h);
  return __dadd_rn(r, l);
}

// ---- a*b mod q, both variable; qinv = RN(1/q); signed result, |r| <= 0.51 q.  |a*b| < 2^88.
__device__ __forceinline__ double mulmod_var(double a, double b, double q, double qinv) {
  double h = __dmul_rn(a, b);
  double l = __fma_rn(a, b, -h);
  double qh = __fma_rn(h, qinv, HML_MAGIC) - HML_MAGIC;
  double r = __fma_rn(-qh, q, h);
  return __dadd_rn(r, l);
}

// ---- Cooley-Tukey (forward) butterfly: (x, y) -> (x + y*w, x - y*w), growth +0.51q per stage.  The twiddle is a
// single double; the quotient estimate comes from h * (1/q) (mulmod_var), so tables and shared memory hold 8 bytes
// per twiddle instead of 16.
__device__ __forceinline__ void ct_butterfly(double &x, double &y, double w, double q, double qinv) {
  double t = mulmod_var(y, w, q, qinv);
  double X = x;
  x = __dadd_rn(X, t);
  y = __dsub_rn(X, t);
}
// ---- Gentleman-Sande (inverse) butterfly: (x, y) -> (x + y, (x - y)*w); x doubles, y resets to <= 0.51q
__device__ __forceinline__ void gs_butterfly(double &x, double &y, double w, double q, double qinv) {
  double d = __dsub_rn(x, y);
  x = __dadd_rn(x, y);
  y = mulmod_var(d, w, q, qinv);
}

// ---- programmatic dependent launch (PDL): every kernel of the library is launched with the programmatic-serialisation
// attribute (launch.h), so its CTAs are scheduled as the CTAs of the previous kernel of the stream exit.  A kernel may touch
// read-only tables (twiddles, moduli, matrices) right away; it must call pdl_wait() before the first access (read OR
// write) to any buffer another kernel may produce or still be reading.  No kernel triggers its dependents early
// (griddepcontrol.launch_dependents): measured on B200 an early trigger lets waiting CTAs of the next kernel take slots
// from the remaining waves of the running one (+5 % on 32-ciphertext chunks); the implicit trigger at CTA exit overlaps
// only the tail and wins everywhere (single hmult 347 -> 297 us, batched 194.7 -> 193.5 us).
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ---- packed limbs.  A residue has at most 36 significant bits, but the ABI word has 64: HBM-bound kernels that hand a limb
// to another kernel of the same op store it "packed" inside the limb's own 8N-byte slot — a plane of N 32-bit low words at
// the start of the slot, a plane of N bytes (bits 32..39) at byte offset 4N — 5 bytes per coefficient instead of 8.  The
// slot geometry (strides, offsets) is unchanged, only 5/8 of it is touched.  i2 = index of a coefficient pair.
__device__ __forceinline__ void st_packed2(u64 *limb_slot, size_t N, size_t i2, u64 a, u64 b) {
  reinterpret_cast<uint2 *>(limb_slot)[i2] = make_uint2((unsigned)a, (unsigned)b);
  reinterpret_cast<unsigned short *>(reinterpret_cast<unsigned char *>(limb_slot) + 4 * N)[i2] =
      (unsigned short)((unsigned)(a >> 32) | ((unsigned)(b >> 32) << 8));
}
// Joins a pair's low words and its two high bytes.  hi is 32 bits wide where the loads are joined right away and 64 bits
// after pin_loads: the casts keep the same instructions for both, with no wider shifts for the 32-bit callers.
template <class H>
__device__ __forceinline__ ulonglong2 packed2_join(uint2 lo, H hi) {
  return make_ulonglong2((u64)(unsigned)(hi & 0xFFu) << 32 | lo.x, (u64)(unsigned)(hi >> 8) << 32 | lo.y);
}
__device__ __forceinline__ ulonglong2 ld_packed2(const u64 *limb_slot, size_t N, size_t i2) {
  const uint2 lo = __ldg(reinterpret_cast<const uint2 *>(limb_slot) + i2);
  const unsigned hi = __ldg(reinterpret_cast<const unsigned short *>(reinterpret_cast<const unsigned char *>(limb_slot) + 4 * N) + i2);
  return packed2_join(lo, hi);
}
// The same two loads, not yet joined, in one 16-byte value (x = the pair's low words, y = its two high bytes): kernels that
// must have every load in flight before the first use hold these in pin_loads, then join them.
__device__ __forceinline__ ulonglong2 ld_packed2_raw(const u64 *limb_slot, size_t N, size_t i2) {
  return make_ulonglong2(__ldg(limb_slot + i2),
                         __ldg(reinterpret_cast<const unsigned short *>(reinterpret_cast<const unsigned char *>(limb_slot) + 4 * N) + i2));
}
__device__ __forceinline__ ulonglong2 packed2_join(ulonglong2 raw) {
  return packed2_join(make_uint2((unsigned)raw.x, (unsigned)(raw.x >> 32)), raw.y);
}

// per-modulus constants kept in device memory
struct ModConst {
  double q;       // modulus as double
  double qinv;    // RN(1/q)
  double ninv;    // N^-1 mod q
  double ninv_q;  // RN(ninv / q)
  u64 qi;         // modulus as integer
  u64 pad;
};

}  // namespace hml
