// Device helpers of the tcgen05 step kernel (pinn_step_tc.cu) and the kernels around it (pinn_reduce.cu, pinn_train.cu).
#pragma once
#include "pinn_common.cuh"
#include "pinn_launch.h"

namespace pinn {

// Per-point stash rows live in shared memory, one row per lane (= point): 64 floats for an MLP warp
// (4 Taylor channels x 16), 32 for the E-net warp.  Rows are NOT padded; instead the column index is
// XOR-swizzled (swz_tc), which keeps float4 groups intact.
constexpr int ROWH = 64;
constexpr int ROWE = 32;
constexpr int EVAL_STASH = 2 * 32 * ROWH;  // floats: Hs + Gs
constexpr int ENET_STASH = 2 * 32 * ROWE;  // floats: E1s + Vs

// Swizzle of the stash: the 16-byte chunk index of a row is XOR-ed with
// s(row) = ((row & 3) << 1) | ((row >> 2) & 1).  Eight consecutive rows get eight different values, so the 128-bit
// accesses of a row by its own lane (quarter-warp = 8 lanes per phase) are conflict-free, and rows r, r+1, r+2, r+3 differ
// in the upper two bits, which keeps the scalar mma.sync fragment loads (8 columns x 4 rows per instruction)
// conflict-free.  Returned in floats (multiple of 4).
__host__ __device__ constexpr int swz_tc(int row) { return ((((row & 3) << 1) | ((row >> 2) & 1)) << 2); }

// ---------------------------------------------------------------------------------------------
// small PTX helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float rcp_approx(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
constexpr float NEG_LOG2E = -1.4426950408889634f;
__device__ __forceinline__ float ex2_approx(float x) {
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x));
  return e;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void named_barrier(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// 3xTF32: x = hi + lo.  The tensor cores read the upper 19 bits of an fp32 operand (they truncate; measured with
// tools/microbench/umma_ts.cu).
//  * weights (split once per CTA by build_weight_image): split_tf32_rn - hi is x ROUNDED to nearest TF32 (add half an
//    ulp, clear the low 13 bits), lo = x - hi is exact in fp32 and gets half an ulp added so that the hardware truncation
//    rounds it to nearest as well: |lo| <= 2^-11 |x| with random sign.
//  * forward-sweep activations: split_tf32_rn3 - the same rounded hi, lo = x - hi left as it is (three instructions): the
//    hardware truncates lo's last one or two bits toward zero, <= 2^-22 |x| and unbiased since lo has a random sign.
//  * reverse-sweep activations and weight-gradient fragments: split_tf32 - two instructions, hi = the 19 bits the hardware would
//    read anyway, lo = x - hi exact (the low 13 mantissa bits; the hardware keeps 11 significant bits of them, i.e. loses
//    at most 2^-22 |x|).  The dropped lo*lo term is <= 2^-21 of the product with the sign of the weight's lo, i.e.
//    unbiased in the mat-vecs; in the weight-gradient contractions (both operands are activations) it is a common factor
//    (1 + ~2^-22) on every term of the sum and cancels like the sum itself does.
__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
  hi = __float_as_uint(x) & 0xffffe000u;
  lo = __float_as_uint(x - __uint_as_float(hi));
}
__device__ __forceinline__ void split_tf32_rn(float x, uint32_t& hi, uint32_t& lo) {
  hi = (__float_as_uint(x) + 0x1000u) & 0xffffe000u;
  lo = __float_as_uint(x - __uint_as_float(hi)) + 0x1000u;
}
__device__ __forceinline__ void split_tf32_rn3(float x, uint32_t& hi, uint32_t& lo) {
  hi = (__float_as_uint(x) + 0x1000u) & 0xffffe000u;
  lo = __float_as_uint(x - __uint_as_float(hi));
}
__device__ __forceinline__ void mma_tf32(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// c += a*b with fp32 accuracy: big*big + big*small + small*big (small*small ~2^-22 dropped)
__device__ __forceinline__ void mma_3xtf32(float (&c)[4], const uint32_t (&ah)[4], const uint32_t (&al)[4],
                                           uint32_t bh0, uint32_t bh1, uint32_t bl0, uint32_t bl1) {
  mma_tf32(c, al, bh0, bh1);
  mma_tf32(c, ah, bl0, bl1);
  mma_tf32(c, ah, bh0, bh1);
}

// packed float32x2 arithmetic (sm_100 FFMA2 / FMUL2 / FADD2): one instruction for two independent values, each rounded
// exactly like its scalar counterpart
__device__ __forceinline__ float2 f2bc(float x) { return make_float2(x, x); }
__device__ __forceinline__ float2 f2neg(float2 a) { return make_float2(-a.x, -a.y); }
__device__ __forceinline__ float2 f2mul(float2 a, float2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ float2 f2add(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 f2fma(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }

// Packed column sums (FADD2 / FFMA2).  Lane = 16 * half + pair
// sums the 16 rows [16 half, 16 half + 16) of the two adjacent columns col2, col2 + 1 (col2 even).  The two halves are
// separate accumulators until the kernel's final fold.
template <int ROW>
__device__ __forceinline__ float2 colsum2(const float* __restrict__ base, int col2, int half) {
  const float* b = base + half * 16 * ROW;
  float2 s0 = make_float2(0.0f, 0.0f), s1 = make_float2(0.0f, 0.0f);
#pragma unroll
  for (int p = 0; p < 16; p += 2) {  // swz_tc(16 half + p) = swz_tc(p): compile-time patterns, [pointer + immediate] loads
    s0 = __fadd2_rn(s0, *reinterpret_cast<const float2*>(b + p * ROW + (col2 ^ swz_tc(p))));
    s1 = __fadd2_rn(s1, *reinterpret_cast<const float2*>(b + (p + 1) * ROW + (col2 ^ swz_tc(p + 1))));
  }
  return __fadd2_rn(s0, s1);
}
// ... and with per-row weights: plain = sum_p v[p][.], weighted = sum_p wgt_p v[p][.] (wgt = the value lane p holds)
template <int ROW>
__device__ __forceinline__ void colsum2_w(const float* __restrict__ base, int col2, int half, float wgt, float2& plain,
                                          float2& weighted) {
  const float* b = base + half * 16 * ROW;
  float2 s0 = make_float2(0.0f, 0.0f), s1 = s0, t0 = s0, t1 = s0;
  const int r0 = half * 16;
#pragma unroll
  for (int p = 0; p < 16; p += 2) {
    const float2 v0 = *reinterpret_cast<const float2*>(b + p * ROW + (col2 ^ swz_tc(p)));
    const float2 v1 = *reinterpret_cast<const float2*>(b + (p + 1) * ROW + (col2 ^ swz_tc(p + 1)));
    const float w0 = __shfl_sync(0xffffffffu, wgt, r0 + p), w1 = __shfl_sync(0xffffffffu, wgt, r0 + p + 1);
    s0 = __fadd2_rn(s0, v0); s1 = __fadd2_rn(s1, v1);
    t0 = __ffma2_rn(v0, make_float2(w0, w0), t0);
    t1 = __ffma2_rn(v1, make_float2(w1, w1), t1);
  }
  plain = __fadd2_rn(s0, s1);
  weighted = __fadd2_rn(t0, t1);
}

// ---------------------------------------------------------------------------------------------
// per-point geometry (poc/main.py:101-108, 269-284; train.py:41-44) and the coefficients of the
// second-order operator D (oracle/closed_form.py:geometry)
// ---------------------------------------------------------------------------------------------
struct Geom {
  float f1, f2, ir1, ir2, al1, al2, al11, al12, al22;
  float R;
};

// raw coordinates of one point, already relative to the two nuclei (5 registers; lets a kernel prefetch the next tile)
struct RawPt {
  float dx1, dx2, y, z, R;
};
__device__ __forceinline__ RawPt load_raw(const StepParams& p, long long i) {
  RawPt r;
  if (p.in_f64) {
    const double xd = ((const double*)p.x)[i], Rd = ((const double*)p.R)[i];
    r.dx1 = (float)(xd - Rd);  // the difference is formed in double so that r near a nucleus keeps its digits
    r.dx2 = (float)(xd + Rd);
    r.y = (float)((const double*)p.y)[i];
    r.z = (float)((const double*)p.z)[i];
    r.R = (float)Rd;
  } else {
    const float xf = ((const float*)p.x)[i];
    r.R = ((const float*)p.R)[i];
    r.dx1 = xf - r.R;
    r.dx2 = xf + r.R;
    r.y = ((const float*)p.y)[i];
    r.z = ((const float*)p.z)[i];
  }
  return r;
}
__device__ __forceinline__ Geom geom_from_raw(const RawPt& r) {
  Geom g;
  const float yz = fmaf(r.y, r.y, r.z * r.z);
  const float q1 = fmaf(r.dx1, r.dx1, yz), q2 = fmaf(r.dx2, r.dx2, yz);
  g.ir1 = rsqrtf(q1);
  g.ir2 = rsqrtf(q2);
  const float r1 = q1 * g.ir1, r2 = q2 * g.ir2;
  g.f1 = __expf(-r1);
  g.f2 = __expf(-r2);
  const float c12 = fmaf(r.dx1, r.dx2, yz) * g.ir1 * g.ir2;
  g.al1 = g.f1 * fmaf(-2.0f, g.ir1, 1.0f);
  g.al2 = g.f2 * fmaf(-2.0f, g.ir2, 1.0f);
  g.al11 = g.f1 * g.f1;
  g.al22 = g.f2 * g.f2;
  g.al12 = 2.0f * g.f1 * g.f2 * c12;
  g.R = r.R;
  return g;
}
__device__ __forceinline__ Geom load_geom(const StepParams& p, long long i) { return geom_from_raw(load_raw(p, i)); }

// ---------------------------------------------------------------------------------------------
// theta (1521 scalars, state_dict order) -> the weight image the step kernel reads (Wts).  Run by `nt` threads
// (t = 0..nt-1) of every CTA, straight into its shared memory.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void build_weight_image(const float* __restrict__ th, Wts* __restrict__ out, int t, int nt) {
  for (int i = t; i < NH; i += nt) {
    const float a = th[O_W1 + 2 * i], b = th[O_W1 + 2 * i + 1];
    out->w0[i] = a; out->w1[i] = b; out->b1[i] = th[O_B1 + i];
    out->ww00[i] = a * a; out->ww01[i] = a * b; out->ww11[i] = b * b;
    out->b2[i] = th[O_B2 + i]; out->wo[i] = th[O_WO + i];
    out->w0s[i] = a * NEG_LOG2E; out->w1s[i] = b * NEG_LOG2E;
    out->b1s[i] = th[O_B1 + i] * NEG_LOG2E; out->b2s[i] = th[O_B2 + i] * NEG_LOG2E;
  }
  for (int i = t; i < NE; i += nt) {
    out->WE1[i] = th[O_WE1 + i]; out->bE1[i] = th[O_BE1 + i];
    out->bE2[i] = th[O_BE2 + i]; out->wE[i] = th[O_WE + i];
    out->WE1s[i] = th[O_WE1 + i] * NEG_LOG2E; out->bE1s[i] = th[O_BE1 + i] * NEG_LOG2E;
    out->bE2s[i] = th[O_BE2 + i] * NEG_LOG2E;
  }
  for (int i = t; i < 12; i += nt) {
    const bool in = i < NL;
    out->WgL[i] = in ? th[O_WGL + i] : 0.0f;
    out->bgL[i] = in ? th[O_BGL + i] : 0.0f;
    out->wg[i] = in ? th[O_WG + i] : 0.0f;
    out->WgLs[i] = in ? th[O_WGL + i] * NEG_LOG2E : 0.0f;
    out->bgLs[i] = in ? th[O_BGL + i] * NEG_LOG2E : 0.0f;
  }
  if (t == 0) { out->bo = th[O_BO]; out->bE = th[O_BE]; out->bg = th[O_BG]; out->pad0 = 0.0f; }
  // ---- tcgen05 operand images: value -> (hi, lo) TF32 pair, round-to-nearest split ----
  auto put = [](float* hi, float* lo, int off, float v) {
    uint32_t h, l;
    split_tf32_rn(v, h, l);
    hi[off] = __uint_as_float(h);
    lo[off] = __uint_as_float(l);
  };
  for (int i = t; i < NH * NH; i += nt) {
    const int j = i / NH, k = i % NH;
    const float wjk = th[O_W2 + i];
    const float a = th[O_W1 + 2 * k], b = th[O_W1 + 2 * k + 1];
    put(out->BS[0], out->BS[1], umma_off(j, k, NH), wjk);
    put(out->BSP[0], out->BSP[1], umma_off(j, k, 2 * NH), wjk * a);
    put(out->BSP[0], out->BSP[1], umma_off(NH + j, k, 2 * NH), wjk * b);
    put(out->BSPP[0], out->BSPP[1], umma_off(j, k, 3 * NH), wjk * (a * a));
    put(out->BSPP[0], out->BSPP[1], umma_off(NH + j, k, 3 * NH), wjk * (a * b));
    put(out->BSPP[0], out->BSPP[1], umma_off(2 * NH + j, k, 3 * NH), wjk * (b * b));
    put(out->BWT[0], out->BWT[1], umma_off(k, j, NH), wjk);
  }
  for (int i = t; i < NE * NE; i += nt) {
    const int j = i / NE, k = i % NE;
    put(out->BE[0], out->BE[1], umma_off(j, k, NE), th[O_WE2 + i]);
    put(out->BET[0], out->BET[1], umma_off(k, j, NE), th[O_WE2 + i]);
  }
}

__device__ __forceinline__ double ld_acquire_gpu(const double* p) {
  double v;
  asm volatile("ld.acquire.gpu.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
  return v;
}

// two sigmoids whose arguments already carry the factor -log2(e) (pre-scaled weights, Wts::w0s ...): 2 MUFU.EX2, one packed
// add, 2 MUFU.RCP
__device__ __forceinline__ float2 sigm2_pre(const float2 up) {
  const float2 d = __fadd2_rn(make_float2(ex2_approx(up.x), ex2_approx(up.y)), make_float2(1.0f, 1.0f));
  return make_float2(rcp_approx(d.x), rcp_approx(d.y));
}

// 1 - s of two sigmoids s = 1/(1+e) as e s.  Where s rounds next to 1 (u > 0) the difference 1 - s keeps only
// e^u 2^-24 of relative accuracy (9e-3 at u = 12), and s(1-s), s'' and s''' inherit it; e s is accurate to a few ulps.
// The product saturates to [0, 1] (FMUL.SAT; there is no packed form), which also turns e = inf, s = 0 (u < -88) into 0
// rather than NaN.
__device__ __forceinline__ float2 one_minus_sigm2(const float2 e, const float2 s) {
  return make_float2(__saturatef(__fmul_rn(e.x, s.x)), __saturatef(__fmul_rn(e.y, s.y)));
}

// sigm2_pre, and 1 - s of both sigmoids (one_minus_sigm2)
__device__ __forceinline__ float2 sigm2_pre(const float2 up, float2& om) {
  const float2 e = make_float2(ex2_approx(up.x), ex2_approx(up.y));
  const float2 d = __fadd2_rn(e, make_float2(1.0f, 1.0f));
  const float2 s = make_float2(rcp_approx(d.x), rcp_approx(d.y));
  om = one_minus_sigm2(e, s);
  return s;
}

// 1 - s of sigmoids s that sigm2_pre formed earlier from the same arguments (the reverse sweeps read s back from the
// stash and form the exponential again)
__device__ __forceinline__ float2 one_minus_sigm2_pre(const float2 up, const float2 s) {
  return one_minus_sigm2(make_float2(ex2_approx(up.x), ex2_approx(up.y)), s);
}

// Q = al11 v1^2 + al12 v1 v2 + al22 v2^2 for two hidden units.  (A 5-operation form v1 (al11 v1 + al12 v2) + al22 v2^2, a
// packed accumulation of N and D, and a non-volatile mma.sync were measured together in round 2: +0.1 % - inside the
// noise - and another rounding pattern at the trained weights; not adopted.)
__device__ __forceinline__ float2 quad_form2(float al11, float al12, float al22, float2 v1, float2 v2) {
  return f2fma(f2mul(f2bc(al11), v1), v1, f2fma(f2mul(f2bc(al12), v1), v2, f2mul(f2mul(f2bc(al22), v2), v2)));
}

#define LD4(ptr) (*reinterpret_cast<const float4*>(ptr))
#define ST4(ptr, a, b, c, d) (*reinterpret_cast<float4*>(ptr) = make_float4(a, b, c, d))

}  // namespace pinn
