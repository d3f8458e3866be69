// Shared host/device helpers for libsurgvid (sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>

#include "../../include/surgvid.h"

namespace sv {

// ---- error plumbing: integer status across the C ABI, message via sv_last_error() ----------------
void set_error(const std::string& msg);
int fail(int code, const std::string& msg);

#define SV_CUDA_OK(expr)                                                                           \
  do {                                                                                             \
    cudaError_t _e = (expr);                                                                       \
    if (_e != cudaSuccess)                                                                         \
      return ::sv::fail(SV_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));          \
  } while (0)

#define SV_CHECK(cond, msg)                                                                        \
  do {                                                                                             \
    if (!(cond)) return ::sv::fail(SV_ERR_INVALID, std::string(msg) + " [" #cond "]");             \
  } while (0)

#define SV_TRY(expr)                                                                               \
  do {                                                                                             \
    int _s = (expr);                                                                               \
    if (_s != SV_OK) return _s;                                                                    \
  } while (0)

inline int launch_status(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(SV_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
  return SV_OK;
}

int device_sm_count();
// opt a kernel in to `bytes` of dynamic shared memory on the CURRENT device (idempotent, thread-safe, failures are not cached)
int ensure_dynamic_smem(const void* fn, int bytes);

typedef __nv_bfloat16 bf16;

// activation codes shared by GEMM epilogue and elementwise kernels
enum Act : int { ACT_NONE = 0, ACT_GELU = 1, ACT_RELU = 2 };

__host__ __device__ inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
__host__ __device__ inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }
__host__ __device__ inline int round_up(int a, int b) { return ceil_div(a, b) * b; }

#ifdef __CUDACC__
// exact (erf) GELU, as nn.GELU() default — mix_transformer_evp.py:33,39
__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f)); }

// GELU(erf) with erf from Abramowitz & Stegun 7.1.26 (|abs err| <= 1.5e-7, far below the bf16 rounding of the result):
// one MUFU.EX2 + one MUFU.RCP instead of erff's branchy polynomial; used where the activation output is stored as bf16.
__device__ __forceinline__ float gelu_erf_fast(float x) {
  const float z = fabsf(x) * 0.70710678118654752440f;
  const float t = __fdividef(1.0f, fmaf(0.3275911f, z, 1.0f));
  float p = fmaf(1.061405429f, t, -1.453152027f);
  p = fmaf(p, t, 1.421413741f);
  p = fmaf(p, t, -0.284496736f);
  p = fmaf(p, t, 0.254829592f);
  const float e = 1.0f - p * t * __expf(-z * z);  // erf(|x|/sqrt2)
  return 0.5f * x * (1.0f + copysignf(e, x));
}

// ---- packed fp32x2 arithmetic (Blackwell FFMA2/FMUL2: two fp32 lanes per instruction) --------------------------------
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 f2_pack(float lo, float hi) { f32x2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void f2_unpack(f32x2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f32x2 f2_fma(f32x2 a, f32x2 b, f32x2 c) { f32x2 r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
__device__ __forceinline__ f32x2 f2_mul(f32x2 a, f32x2 b) { f32x2 r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
// two bf16 packed in a 32-bit word -> fp32x2 (exact: bf16 is the top half of an fp32)
__device__ __forceinline__ f32x2 f2_from_bf16x2(uint32_t v) {
  f32x2 r;
  // prmt/and run on the integer ALU; a plain shift is often emitted as IMAD.U32, which competes with the FFMA2s for the FMA pipe
  asm("{\n\t.reg .b32 lo, hi;\n\tprmt.b32 lo, %1, 0, 0x1044;\n\tand.b32 hi, %1, 0xffff0000;\n\tmov.b64 %0, {lo, hi};\n\t}" : "=l"(r) : "r"(v));
  return r;
}

// GELU(erf) for two lanes without MUFU.  erf is odd, so with xc = clamp(x, -lim, lim) and w = xc^2:
//   erf(x/sqrt2) ~= (xc/sqrt2) * P(w/2),   P = degree-8 near-minimax fit of erf(z)/z on z in [0,3] (|erf err| <= 1.7e-5),
//   and   y = 0.5*x*(1 + erf(x/sqrt2)) = 0.5*x + x * (xc * Q(w)),
// Q(w) = 0.5/sqrt2 * P(w/2) with the constant factors folded into the coefficients.  |GELU error| <= 6.1e-5 absolute —
// below the bf16 rounding of the stored result for |y| > 0.03 and negligible below that (end-to-end parity unchanged).
// lim = 4.244771 (z = 3.0015, just past the fit's end, where P crosses 1) is an fp32 value at which the fp32 evaluation of
// xc * Q(w) is exactly 0.5: beyond the clamp y is exactly x or 0, so the error does not grow with |x| (at 3*sqrt2 it was
// 0.5 - 2.4e-6, an error of 2.4e-6 |x|).  |xc * Q| <= 0.5, so x * (xc * Q) cannot overflow for any finite x
// ((x * xc) * Q did for |x| >= 8.0e37).
__device__ __forceinline__ f32x2 f2_gelu_erf_poly(f32x2 x) {
  float x0, x1;
  f2_unpack(x, x0, x1);
  const float lim = 4.244771f;  // see above: fp32 xc * Q(w) == 0.5 exactly
  const f32x2 xc = f2_pack(fminf(fmaxf(x0, -lim), lim), fminf(fmaxf(x1, -lim), lim));
  const f32x2 w = f2_mul(xc, xc);
#define SV_C2(v) f2_pack(v, v)
  // q_k = c_k * 0.5^k * 0.5/sqrt2,  c_k from the fit of erf(z) = z * sum c_k z^(2k)
  f32x2 q = f2_fma(SV_C2(5.626770213e-11f), w, SV_C2(-5.371870724e-09f));
  q = f2_fma(q, w, SV_C2(2.268296714e-07f));
  q = f2_fma(q, w, SV_C2(-5.646215765e-06f));
  q = f2_fma(q, w, SV_C2(9.359063167e-05f));
  q = f2_fma(q, w, SV_C2(-1.109400333e-03f));
  q = f2_fma(q, w, SV_C2(9.818119241e-03f));
  q = f2_fma(q, w, SV_C2(-6.634692395e-02f));
  q = f2_fma(q, w, SV_C2(3.989031282e-01f));
  return f2_fma(x, f2_mul(xc, q), f2_mul(x, SV_C2(0.5f)));
#undef SV_C2
}

// Two independent GELU evaluations with their Horner chains interleaved step by step (the dependent FFMA2 chain of one
// evaluation leaves issue slots empty; two side by side fill them).
__device__ __forceinline__ void f2_gelu_erf_poly_x2(f32x2& xa, f32x2& xb) {
  float a0, a1, b0, b1;
  f2_unpack(xa, a0, a1);
  f2_unpack(xb, b0, b1);
  const float lim = 4.244771f;
  const f32x2 ca = f2_pack(fminf(fmaxf(a0, -lim), lim), fminf(fmaxf(a1, -lim), lim));
  const f32x2 cb = f2_pack(fminf(fmaxf(b0, -lim), lim), fminf(fmaxf(b1, -lim), lim));
  const f32x2 wa = f2_mul(ca, ca), wb = f2_mul(cb, cb);
#define SV_C2(v) f2_pack(v, v)
  f32x2 qa = f2_fma(SV_C2(5.626770213e-11f), wa, SV_C2(-5.371870724e-09f));
  f32x2 qb = f2_fma(SV_C2(5.626770213e-11f), wb, SV_C2(-5.371870724e-09f));
#define SV_STEP(c) qa = f2_fma(qa, wa, SV_C2(c)); qb = f2_fma(qb, wb, SV_C2(c));
  SV_STEP(2.268296714e-07f)
  SV_STEP(-5.646215765e-06f)
  SV_STEP(9.359063167e-05f)
  SV_STEP(-1.109400333e-03f)
  SV_STEP(9.818119241e-03f)
  SV_STEP(-6.634692395e-02f)
  SV_STEP(3.989031282e-01f)
#undef SV_STEP
  xa = f2_fma(xa, f2_mul(ca, qa), f2_mul(xa, SV_C2(0.5f)));
  xb = f2_fma(xb, f2_mul(cb, qb), f2_mul(xb, SV_C2(0.5f)));
#undef SV_C2
}

// four independent evaluations, Horner steps in lockstep (used where only two warps share a scheduler)
__device__ __forceinline__ void f2_gelu_erf_poly_x4(f32x2& xa, f32x2& xb, f32x2& xc, f32x2& xd) {
  const float lim = 4.244771f;
  auto clamp2 = [&](f32x2 v) {
    float v0, v1;
    f2_unpack(v, v0, v1);
    return f2_pack(fminf(fmaxf(v0, -lim), lim), fminf(fmaxf(v1, -lim), lim));
  };
  const f32x2 ca = clamp2(xa), cb = clamp2(xb), cc = clamp2(xc), cd = clamp2(xd);
  const f32x2 wa = f2_mul(ca, ca), wb = f2_mul(cb, cb), wc = f2_mul(cc, cc), wd = f2_mul(cd, cd);
#define SV_C2(v) f2_pack(v, v)
  f32x2 qa = f2_fma(SV_C2(5.626770213e-11f), wa, SV_C2(-5.371870724e-09f));
  f32x2 qb = f2_fma(SV_C2(5.626770213e-11f), wb, SV_C2(-5.371870724e-09f));
  f32x2 qc = f2_fma(SV_C2(5.626770213e-11f), wc, SV_C2(-5.371870724e-09f));
  f32x2 qd = f2_fma(SV_C2(5.626770213e-11f), wd, SV_C2(-5.371870724e-09f));
#define SV_STEP(c) qa = f2_fma(qa, wa, SV_C2(c)); qb = f2_fma(qb, wb, SV_C2(c)); qc = f2_fma(qc, wc, SV_C2(c)); qd = f2_fma(qd, wd, SV_C2(c));
  SV_STEP(2.268296714e-07f)
  SV_STEP(-5.646215765e-06f)
  SV_STEP(9.359063167e-05f)
  SV_STEP(-1.109400333e-03f)
  SV_STEP(9.818119241e-03f)
  SV_STEP(-6.634692395e-02f)
  SV_STEP(3.989031282e-01f)
#undef SV_STEP
  xa = f2_fma(xa, f2_mul(ca, qa), f2_mul(xa, SV_C2(0.5f)));
  xb = f2_fma(xb, f2_mul(cb, qb), f2_mul(xb, SV_C2(0.5f)));
  xc = f2_fma(xc, f2_mul(cc, qc), f2_mul(xc, SV_C2(0.5f)));
  xd = f2_fma(xd, f2_mul(cd, qd), f2_mul(xd, SV_C2(0.5f)));
#undef SV_C2
}

// GELU(erf) through the MUFU pipe, two lanes:  y = x * sigmoid(2 g(x)),  g(x) = x (c0 + c1 x^2 + c2 x^4) ~= atanh(erf(x / sqrt2))
// (least-squares fit of the GELU itself on [-6, 6]: |GELU error| <= 3.0e-5 absolute, |erf error| <= 1.2e-4; x^2 is clamped at 49 where
// the sigmoid has long saturated).  sigmoid = 1 / (1 + 2^t) with t = x * q(x^2), q = -2 log2(e) (c0 + c1 u + c2 u^2): one MUFU.EX2 and one
// MUFU.RCP per element (relative error ~1e-6 each) and 6 FMA-pipe instructions per PAIR, against 13 for the MUFU-free polynomial —
// the depthwise-conv kernel is bound by the FMA pipe, and the MUFU pipe is otherwise idle there.
__device__ __forceinline__ float sv_ex2(float x) { float r; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float sv_rcp(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float sv_tanh(float x) { float r; asm("tanh.approx.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ f32x2 f2_add(f32x2 a, f32x2 b) { f32x2 r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
#define SV_GELU_G0 0.7974584707822386f
#define SV_GELU_G1 0.03705034510045914f
#define SV_GELU_G2 (-0.0003587323611556633f)
__device__ __forceinline__ f32x2 f2_gelu_sigmoid(f32x2 x) {
  const float k = -2.8853900817779268f;   // -2 log2(e)
  f32x2 u = f2_mul(x, x);
  float u0, u1;
  f2_unpack(u, u0, u1);
  u = f2_pack(fminf(u0, 49.f), fminf(u1, 49.f));
  f32x2 q = f2_fma(u, f2_pack(k * SV_GELU_G2, k * SV_GELU_G2), f2_pack(k * SV_GELU_G1, k * SV_GELU_G1));
  q = f2_fma(q, u, f2_pack(k * SV_GELU_G0, k * SV_GELU_G0));
  float t0, t1;
  f2_unpack(f2_mul(x, q), t0, t1);
  const f32x2 d = f2_add(f2_pack(sv_ex2(t0), sv_ex2(t1)), f2_pack(1.f, 1.f));
  float d0, d1;
  f2_unpack(d, d0, d1);
  return f2_mul(x, f2_pack(sv_rcp(d0), sv_rcp(d1)));
}
// same g(x), but y = 0.5 x (1 + tanh(g)): ONE MUFU per element; tanh.approx carries ~2^-11 relative error, i.e. up to ~2.5e-4 |x|
// absolute on the result (worst in the negative tail, where 1 + tanh cancels)
__device__ __forceinline__ f32x2 f2_gelu_tanh(f32x2 x) {
  f32x2 u = f2_mul(x, x);
  float u0, u1;
  f2_unpack(u, u0, u1);
  u = f2_pack(fminf(u0, 49.f), fminf(u1, 49.f));
  f32x2 q = f2_fma(u, f2_pack(SV_GELU_G2, SV_GELU_G2), f2_pack(SV_GELU_G1, SV_GELU_G1));
  q = f2_fma(q, u, f2_pack(SV_GELU_G0, SV_GELU_G0));
  float t0, t1;
  f2_unpack(f2_mul(x, q), t0, t1);
  const f32x2 hx = f2_mul(x, f2_pack(0.5f, 0.5f));
  return f2_fma(hx, f2_pack(sv_tanh(t0), sv_tanh(t1)), hx);
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ float2 unpack_bf16x2(uint32_t v) {
  __nv_bfloat162 t = *reinterpret_cast<__nv_bfloat162*>(&v);
  return __bfloat1622float2(t);
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
#endif

}  // namespace sv
