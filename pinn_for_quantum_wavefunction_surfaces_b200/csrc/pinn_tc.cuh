// tcgen05 / TMEM / mbarrier helpers and the TMEM column map shared by the tcgen05 step kernels
// (pinn_step_tc.cu: one warp per 32-point row and role).
#pragma once
#include "pinn_device.cuh"

namespace pinn {

// ---------------------------------------------------------------------------------------------
// tcgen05 / TMEM / mbarrier PTX
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// tcgen05.wait::ld that also "touches" the loaded registers: their consumers cannot be scheduled above the wait, and no
// memory clobber is needed (shared-memory loads of weights may move freely around the TMEM traffic)
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tc_wait_ld(float (&v)[N]) {
  static_assert(N == 8 || N == 16, "8 or 16 registers");
  if constexpr (N == 8)
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+f"(v[0]), "+f"(v[1]), "+f"(v[2]), "+f"(v[3]), "+f"(v[4]), "+f"(v[5]), "+f"(v[6]), "+f"(v[7]));
  else
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+f"(v[0]), "+f"(v[1]), "+f"(v[2]), "+f"(v[3]), "+f"(v[4]), "+f"(v[5]), "+f"(v[6]), "+f"(v[7]), "+f"(v[8]),
                   "+f"(v[9]), "+f"(v[10]), "+f"(v[11]), "+f"(v[12]), "+f"(v[13]), "+f"(v[14]), "+f"(v[15]));
}

__device__ __forceinline__ void tc_mma(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}
// one lane of a fully converged warp (the branch around it must be warp-uniform)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tc_commit(uint32_t mbar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(mbar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t mbar, uint32_t parity) {
  uint32_t done = 0;
  while (!done) {
    asm volatile(
        "{\n\t.reg .pred q;\n\tmbarrier.try_wait.parity.shared::cta.b64 q, [%1], %2;\n\tselp.u32 %0, 1, 0, q;\n\t}"
        : "=r"(done)
        : "r"(mbar), "r"(parity)
        : "memory");
  }
}
// shared-memory operand descriptor: K-major, no swizzle, N rows (see umma_off): LBO = 128*(N/8) B, SBO = 128 B
__device__ __forceinline__ uint64_t tc_bdesc(uint32_t saddr, uint32_t N) {
  return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)N << 16) | ((uint64_t)8 << 32) | ((uint64_t)1 << 46);
}
// instruction descriptor: D = f32, A = B = tf32, both K-major, M = 128
__host__ __device__ constexpr uint32_t tc_idesc(uint32_t N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((N >> 3) << 17) | ((128u >> 4) << 24);
}
// D (+)= (a_hi + a_lo) * (B_hi + B_lo) without the lo*lo term
__device__ __forceinline__ void tc_mma3(uint32_t d, uint32_t a_hi, uint32_t a_lo, uint32_t b_hi, uint32_t b_lo, uint32_t N,
                                        uint32_t idesc, bool first) {
  tc_mma(d, a_lo, tc_bdesc(b_hi, N), idesc, first ? 0u : 1u);
  tc_mma(d, a_hi, tc_bdesc(b_lo, N), idesc, 1u);
  tc_mma(d, a_hi, tc_bdesc(b_hi, N), idesc, 1u);
}

__device__ __forceinline__ void tc_st16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
               "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
               "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]));
}
__device__ __forceinline__ void tc_ld8(uint32_t taddr, float (&v)[8]) {
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
#pragma unroll
  for (int i = 0; i < 8; i++) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tc_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
#pragma unroll
  for (int i = 0; i < 16; i++) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tc_st4f(uint32_t taddr, float a, float b, float c, float d) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" ::"r"(taddr), "r"(__float_as_uint(a)),
               "r"(__float_as_uint(b)), "r"(__float_as_uint(c)), "r"(__float_as_uint(d)));
}
__device__ __forceinline__ void tc_st16f(uint32_t taddr, const float (&x)[16]) {
  uint32_t v[16];
#pragma unroll
  for (int i = 0; i < 16; i++) v[i] = __float_as_uint(x[i]);
  tc_st16(taddr, v);
}
__device__ __forceinline__ void tc_st8(uint32_t taddr, const uint32_t (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "r"(v[0]), "r"(v[1]),
               "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]));
}
__device__ __forceinline__ void tc_st8f(uint32_t taddr, const float (&x)[8]) {
  uint32_t v[8];
#pragma unroll
  for (int i = 0; i < 8; i++) v[i] = __float_as_uint(x[i]);
  tc_st8(taddr, v);
}
// truncating split of 8 values, stored as hi / lo halves (reverse sweep)
__device__ __forceinline__ void tc_st_split8(uint32_t t_hi, uint32_t t_lo, const float (&x)[8]) {
  uint32_t hi[8], lo[8];
#pragma unroll
  for (int i = 0; i < 8; i++) split_tf32(x[i], hi[i], lo[i]);
  tc_st8(t_hi, hi);
  tc_st8(t_lo, lo);
}
// split 16 values and store them as the hi / lo halves of an A operand row.  RN: the round-to-nearest split of the
// activations (three instructions, split_tf32_rn3: measured as accurate as the four-instruction form, -1.5 % time; forward
// sweep: psi ~ 2e-5 at the boundary is a cancellation of O(0.1) terms, a common rounding direction of all points would
// add up in the loss and its gradient); otherwise the two-instruction truncating split (reverse sweep: a common factor
// 1 - O(2^-22) on a gradient is harmless).  See split_tf32 in pinn_device.cuh.
template <bool RN>
__device__ __forceinline__ void tc_st_split16(uint32_t t_hi, uint32_t t_lo, const float (&x)[16]) {
  uint32_t hi[16], lo[16];
#pragma unroll
  for (int i = 0; i < 16; i++) {
    if (RN) split_tf32_rn3(x[i], hi[i], lo[i]);
    else split_tf32(x[i], hi[i], lo[i]);
  }
  tc_st16(t_hi, hi);
  tc_st16(t_lo, lo);
}

// ---------------------------------------------------------------------------------------------
// TMEM column map (512 columns x 128 lanes; lane = point of the super-tile)
//   MLP role r (r = 0,1): columns [192 r, 192 r + 192)
//     forward : A = s hi|s' hi|s'' hi|s lo|s' lo|s'' lo (6 x 16)   D = V0 (16) | V1,V2 (32) | P00,P01,P11 (48)
//     reverse : A = vbar hi (4 x 16) | vbar lo (4 x 16)            D = hbar (4 x 16)
//   E-net role: columns [384, 480): A = e1 / vbar hi (32) | lo (32), D (32); between the forward's read of D and the
//               reverse MMA, D holds s'(1-s) of layer 2 for the reverse sweep
//   E-net role, forward to reverse: columns [480, 512): s'(1-s) of layer 1 for the reverse sweep
// ---------------------------------------------------------------------------------------------
constexpr uint32_t TC_MLP_COLS = 192, TC_E_BASE = 384, TC_SP_PARK = 480;
constexpr uint32_t F_S_HI = 0, F_SP_HI = 16, F_SPP_HI = 32, F_S_LO = 48, F_SP_LO = 64, F_SPP_LO = 80;
constexpr uint32_t F_V0 = 96, F_V12 = 112, F_P = 144;
constexpr uint32_t B_VB_HI = 0, B_VB_LO = 64, B_HB = 128;
constexpr uint32_t E_A_HI = 0, E_A_LO = 32, E_D = 64;

constexpr int COORD_COL_BYTES = 128 * 8;                      // one coordinate column of a super-tile (float64 worst case)
constexpr int COORD_STAGE_BYTES = 4 * COORD_COL_BYTES + 128 * 4;  // + one word per point for the set mask
constexpr int COORD_STAGES = 2;  // the coordinate stage runs one super-tile ahead

struct TcCtx {
  uint32_t tbase;      // TMEM base address of the allocation
  uint32_t tlane;      // tbase + (32 * group) << 16: this warp's lane quarter
  uint32_t mbar;       // shared address of this role's mbarrier
  uint32_t phase;      // parity of the next completion
  int bar_id;          // named barrier of this role (128 threads)
  bool issuer;         // this WARP issues the role's MMAs (warp-uniform; one elected lane does it, so that the operand
                       // addresses stay in uniform registers and no per-thread broadcast loop is generated)
  uint32_t wts_saddr;  // shared address of the weight image
  int tl_it;           // tile counter (debug timeline builds)
};

__device__ __forceinline__ void tc_wait_mma(TcCtx& c) {
  mbar_wait(c.mbar, c.phase);
  c.phase ^= 1u;
  tc_fence_after();
}


// coordinates of point `i`: from the caller's arrays, or generated from the grid descriptor (meshgrid 'ij' order;
// positions are formed in double like the reference's linspace and rounded once, the nucleus offsets before rounding)
__device__ __forceinline__ void grid_ijk(const GridDesc& g, long long i, int& ix, int& iy, int& iz) {
  if ((unsigned long long)i < 0x80000000ull) {  // every practical grid (464^3 = 1.0e8): 32-bit divisions, a fifth of the code
    const unsigned u = (unsigned)i, nz = (unsigned)g.nz, ny = (unsigned)g.ny;
    const unsigned r = u / nz;
    iz = (int)(u - r * nz);
    const unsigned q = r / ny;
    iy = (int)(r - q * ny);
    ix = (int)q;
    return;
  }
  iz = (int)(i % g.nz);
  const long long r = i / g.nz;
  iy = (int)(r % g.ny);
  ix = (int)(r / g.ny);
}
__device__ __forceinline__ RawPt tc_grid_point(const StepParams& p, long long i) {
  int ix, iy, iz;
  grid_ijk(p.grid, i, ix, iy, iz);
  const double x = fma((double)ix, p.grid.dx, p.grid.x0);
  RawPt r;
  r.dx1 = (float)(x - p.grid.R);
  r.dx2 = (float)(x + p.grid.R);
  r.y = (float)fma((double)iy, p.grid.dy, p.grid.y0);
  r.z = (float)fma((double)iz, p.grid.dz, p.grid.z0);
  r.R = (float)p.grid.R;
  return r;
}

// Spheroidal sweep (GridDesc::sph): point i -> R index k and node indices (is, jn); pad = a slot behind the R's ns*nnu
// nodes (it repeats the last node, so that it is finite, and gets weight 0).  The launcher keeps every index below 2^31.
__device__ __forceinline__ void sph_index(const GridDesc& g, long long i, int& k, int& is, int& jn, bool& pad) {
  const unsigned u = (unsigned)i, per = (unsigned)g.tiles_per_R * 128u, nn = (unsigned)(g.ns * g.nnu), nnu = (unsigned)g.nnu;
  k = (int)(u / per);
  unsigned l = u - (unsigned)k * per;
  pad = l >= nn;
  if (pad) l = nn - 1;
  is = (int)(l / nnu);
  jn = (int)(l - (unsigned)is * nnu);
}
// x = R (1 + s/R) nu, y = sqrt(s (2R + s) (1 - nu^2)), z = 0: every operation in double, rounded as written (the _rn
// intrinsics forbid contraction into FMAs), so that a host that evaluates the same expressions gets the same points;
// s (2R + s) is R^2 (mu^2 - 1) without the cancellation near the axis
__device__ __forceinline__ RawPt tc_sph_point(const GridDesc& g, long long i) {
  int k, is, jn;
  bool pad;
  sph_index(g, i, k, is, jn, pad);
  const double R = g.Rs[k], s = g.s[is], nu = g.nu[jn];
  const double x = __dmul_rn(__dmul_rn(R, __dadd_rn(1.0, __ddiv_rn(s, R))), nu);
  RawPt r;
  r.dx1 = (float)__dsub_rn(x, R);
  r.dx2 = (float)__dadd_rn(x, R);
  r.y = (float)__dsqrt_rn(__dmul_rn(__dmul_rn(s, __dadd_rn(__dmul_rn(2.0, R), s)), __dsub_rn(1.0, __dmul_rn(nu, nu))));
  r.z = 0.0f;
  r.R = (float)R;
  return r;
}
// quadrature weight of point i: 2 pi ws wnu r1 r2 with r1 r2 = (R + s)^2 - (R nu)^2 (the volume element in (s, nu, phi)),
// 0 for a padding slot
__device__ __forceinline__ double sph_weight(const GridDesc& g, long long i) {
  int k, is, jn;
  bool pad;
  sph_index(g, i, k, is, jn, pad);
  const double R = g.Rs[k], s = g.s[is], nu = g.nu[jn];
  const double rs = R + s, rn = R * nu;
  return pad ? 0.0 : 6.283185307179586 * g.ws[is] * g.wnu[jn] * (rs * rs - rn * rn);
}

}  // namespace pinn
