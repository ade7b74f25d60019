// Fused PINN residual-and-gradient kernel, tcgen05 engine (B200, sm_100a).
//
// oracle/closed_form.py is the specification; poc/main.py:247-303, 82-120, 341-355 and train.py:41-57 are what it
// replaces.  The four mat-vec families of a tile
//     base-MLP layer 2 forward      V = W2 h        (4 Taylor channels)
//     base-MLP layer 2 reverse      hbar = W2^T vbar (4 channels)
//     E-net layer 2 forward / reverse (32 x 32)
// run on the 5th-generation tensor cores instead of FFMA chains:
//   * a CTA works on a SUPER-TILE of 128 collocation points: 4 groups x 32 points, thread = point =
//     TMEM lane.  Warps are specialised by role (one warpgroup per MLP evaluation, one for
//     E-net + gate); the 4 warps of a role form the 128 rows of an M=128 tcgen05.mma.
//   * every thread writes its row of the A operand (activations, split x = hi + lo with hi = the 19 bits
//     the tensor core reads) straight from registers into TENSOR MEMORY with tcgen05.st; the B operands
//     (weights, split the same way, canonical K-major layout) sit in shared memory, built once per CTA:
//     theta arrives by one TMA bulk copy (or inside the kernel parameters, INLINE) and all threads turn it
//     into the operand images (build_weight_image); D accumulates in TMEM and comes back with tcgen05.ld.
//     3xTF32 (lo*hi + hi*lo + hi*hi) keeps fp32 accuracy (tools/microbench/umma_ts.cu: 4e-7 relative).
//   * the forward uses the linearity of the Taylor channels in the layer-1 quantities: with A = {s, s', s''}
//     (3 x 16 columns instead of 4 x 16) and the pre-multiplied operand images BS/BSP/BSPP the 4-channel
//     product needs 18 instead of 24 MMAs.
//   * an M=128, K=8 TF32 MMA costs ~47 cycles for any N <= 64 (measured), so the tensor pipe is busy
//     ~40 cycles per point and overlaps the element-wise work of the other roles; the weight-gradient
//     contractions (K = points) stay on mma.sync, reading the shared-memory stash, and are issued while
//     the reverse-sweep MMAs are in flight.
//   * coordinates travel global -> shared with cp.async one super-tile ahead (page-locked host memory
//     works as a source); the kernel is launched as a programmatic dependent of the kernel in front of it;
//     the code after the common set-up exists once per kind of role (MLP / E-net) and, in the poc training
//     kernel, starts with setmaxnreg (the E-net warpgroup lends registers to the two MLP warpgroups).
#include <cstring>
#include <type_traits>

#include "pinn_tc.cuh"

// Debug builds only (-DPINN_TIMELINE, tools/timeline.py): warp-level clock64() stamps at the phase boundaries of one
// super-tile of CTA 0, to see where a tile's time goes.  Not compiled into the product library.
#ifdef PINN_TIMELINE
__device__ long long g_timeline[16 * 32];
#define TL(i) do { if (blockIdx.x == 0 && c.tl_it == 3 && (threadIdx.x & 31) == 0) g_timeline[(threadIdx.x >> 5) * 32 + (i)] = clock64(); } while (0)
extern "C" int pinn_debug_timeline(long long* out) { return (int)cudaMemcpyFromSymbol(out, g_timeline, sizeof(g_timeline)); }
// whole-kernel stamps of warp 0 of CTA 0: [0] entry, [1] setup done, [2 + it] start of its it-th super-tile, [40] loop done, [41] end
__device__ long long g_timeline_k[48];
__device__ long long g_timeline_cta[2 * 256];  // per CTA: globaltimer (ns) at entry and at exit
extern "C" int pinn_debug_timeline_cta(long long* out) { return (int)cudaMemcpyFromSymbol(out, g_timeline_cta, sizeof(g_timeline_cta)); }
#define TLK(i) do { if (blockIdx.x == 0 && threadIdx.x == 0) g_timeline_k[(i)] = clock64(); \
                    if (threadIdx.x == 0 && ((i) == 0 || (i) == 41)) { unsigned long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); \
                      g_timeline_cta[blockIdx.x * 2 + ((i) == 41)] = (long long)t_; } } while (0)
extern "C" int pinn_debug_timeline_kernel(long long* out) { return (int)cudaMemcpyFromSymbol(out, g_timeline_k, sizeof(g_timeline_k)); }
#else
#define TL(i) do { } while (0)
#define TLK(i) do { } while (0)
#endif

namespace pinn {


template <int NEV>
__host__ __device__ constexpr int tc_group_stash_floats() { return NEV * EVAL_STASH + ENET_STASH; }
// geometry hand-off: the E-net warp of a group computes the per-point geometry once and publishes it to the group's MLP
// warps: 12 floats per point {f1, f2, ir1, ir2 | al1, al2, al11, al12 | al22, dx1, dx2, set bits}, two buffers
constexpr int GEO_BYTES = 2 * 128 * 12 * 4;
template <int NEV>
__host__ __device__ constexpr size_t tc_smem_bytes() {
  return sizeof(Wts) + 64 /*mbarriers + tmem base*/ + sizeof(float2) * 4 * 2 * 3 * 32 + sizeof(float) * 4 * tc_group_stash_floats<NEV>() +
         COORD_STAGES * COORD_STAGE_BYTES + GEO_BYTES;
}

// ---------------------------------------------------------------------------------------------
// coordinate stage: the x,y,z,R (and set mask) of the NEXT super-tile travel global -> shared with cp.async while the
// current one is computed, so that no register (and no warp) waits for them.  This is what lets the host entry hand
// the kernel page-locked host memory: the PCIe round trip is hidden behind a whole tile of work.
//   buffer = 4 columns x 128 points x 8 B (float64 inputs; float32 use the first half of each column) + 128 mask words
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void cp_async4(uint32_t dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async8(uint32_t dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// issued by the E-net warp of a group for the group's 32 points (slot = 32 * group + lane of the super-tile)
__device__ __forceinline__ void coord_stage_issue(const StepParams& p, unsigned char* buf, int slot, long long i) {
  const uint32_t b = smem_u32(buf);
  if (p.in_f64) {
    cp_async8(b + 0 * COORD_COL_BYTES + slot * 8, (const double*)p.x + i);
    cp_async8(b + 1 * COORD_COL_BYTES + slot * 8, (const double*)p.y + i);
    cp_async8(b + 2 * COORD_COL_BYTES + slot * 8, (const double*)p.z + i);
    cp_async8(b + 3 * COORD_COL_BYTES + slot * 8, (const double*)p.R + i);
  } else {
    cp_async4(b + 0 * COORD_COL_BYTES + slot * 4, (const float*)p.x + i);
    cp_async4(b + 1 * COORD_COL_BYTES + slot * 4, (const float*)p.y + i);
    cp_async4(b + 2 * COORD_COL_BYTES + slot * 4, (const float*)p.z + i);
    cp_async4(b + 3 * COORD_COL_BYTES + slot * 4, (const float*)p.R + i);
  }
  // the aligned 4-byte word that holds mask[i] (allocations are at least 4-byte granular); the reader picks the byte
  if (p.mask) cp_async4(b + 4 * COORD_COL_BYTES + slot * 4, (const void*)((uintptr_t)(p.mask + i) & ~(uintptr_t)3));
}
// Full super-tiles of 16-byte aligned columns travel as FIVE bulk copies (cp.async.bulk, the TMA engine) issued by one
// thread: 512 B (float32) or 1 KB (float64) per column plus 128 mask bytes, completing on the stage's mbarrier.  Over
// PCIe (page-locked host inputs read in place) the bus then sees a few large reads per super-tile instead of the 16 + 4
// 128-byte requests of the per-lane path, which all 148 CTAs used to issue in bursts at their tile boundaries; the
// per-lane path remains for the ragged last super-tile and for unaligned columns.
__device__ __forceinline__ void coord_stage_issue_bulk(const StepParams& p, unsigned char* buf, uint64_t* bar, long long st) {
  const uint32_t b = smem_u32(buf), mb = smem_u32(bar);
  const uint32_t colb = p.in_f64 ? 1024u : 512u;
  const uint32_t total = 4u * colb + (p.mask ? 128u : 0u);
  // the buffer was last READ through the generic proxy (by every warp, two super-tiles ago; ordered before this point
  // by the role / group barriers): order those reads before the async-proxy writes
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mb), "r"(total) : "memory");
  const char* src[4] = {(const char*)p.x, (const char*)p.y, (const char*)p.z, (const char*)p.R};
#pragma unroll
  for (int c = 0; c < 4; c++)
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(b + c * COORD_COL_BYTES),
                 "l"(src[c] + (size_t)st * colb), "r"(colb), "r"(mb)
                 : "memory");
  if (p.mask)
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(b + 4 * COORD_COL_BYTES),
                 "l"(p.mask + (size_t)st * 128), "r"(128u), "r"(mb)
                 : "memory");
}
__device__ __forceinline__ RawPt coord_stage_read(const StepParams& p, const unsigned char* buf, int slot) {
  RawPt r;
  if (p.in_f64) {
    const double xd = *(const double*)(buf + 0 * COORD_COL_BYTES + slot * 8), Rd = *(const double*)(buf + 3 * COORD_COL_BYTES + slot * 8);
    r.dx1 = (float)(xd - Rd);  // the difference is formed in double so that r near a nucleus keeps its digits
    r.dx2 = (float)(xd + Rd);
    r.y = (float)*(const double*)(buf + 1 * COORD_COL_BYTES + slot * 8);
    r.z = (float)*(const double*)(buf + 2 * COORD_COL_BYTES + slot * 8);
    r.R = (float)Rd;
  } else {
    const float xf = *(const float*)(buf + 0 * COORD_COL_BYTES + slot * 4);
    r.R = *(const float*)(buf + 3 * COORD_COL_BYTES + slot * 4);
    r.dx1 = xf - r.R;
    r.dx2 = xf + r.R;
    r.y = *(const float*)(buf + 1 * COORD_COL_BYTES + slot * 4);
    r.z = *(const float*)(buf + 2 * COORD_COL_BYTES + slot * 4);
  }
  return r;
}

__device__ __forceinline__ void tc_role_sync(const TcCtx& c) {
  tc_wait_st();
  tc_fence_before();
  // Only the issuing warp has to know that all four warps' operand rows are in tensor memory: it syncs, the other three
  // signal and go on (their next use of the result waits on the MMA's mbarrier anyway; their stash rows are their own).
  // v15: step -1.1 %, same bits (profiles/r02_ar_ab_role_barrier_arrive.log).  Choosing the issuer dynamically - the first
  // warp to arrive, or the last one with no barrier at all - measured 1.6 % / 2.7 % SLOWER than the fixed one (r02_as_*).
  if (c.issuer) named_barrier(c.bar_id, 128);
  else asm volatile("bar.arrive %0, %1;" ::"r"(c.bar_id), "r"(128) : "memory");
}

// ---------------------------------------------------------------------------------------------
// base MLP, forward (oracle/closed_form.py:mlp_fwd)
// ---------------------------------------------------------------------------------------------
template <bool STASH>
__device__ __forceinline__ void tc_mlp_forward(const Wts& w, TcCtx& c, uint32_t cb, float a, float b, float al1, float al2,
                                               float al11, float al12, float al22, float* __restrict__ Hrow,
                                               float* __restrict__ Grow, int sx, float& Nv, float& Dv) {
  float s_[NH], sp_[NH], spp_[NH];
#pragma unroll
  for (int k4 = 0; k4 < NH; k4 += 4) {
    const float4 w0v = LD4(&w.w0s[k4]), w1v = LD4(&w.w1s[k4]), b1v = LD4(&w.b1s[k4]);  // times -log2(e)
    const float w0a[4] = {w0v.x, w0v.y, w0v.z, w0v.w}, w1a[4] = {w1v.x, w1v.y, w1v.z, w1v.w};
    const float b1a[4] = {b1v.x, b1v.y, b1v.z, b1v.w};
#pragma unroll
    for (int i = 0; i < 4; i += 2) {  // two hidden units per instruction; u = -log2(e) * pre-activation, one rounding
      const float2 u = f2fma(f2bc(a), make_float2(w0a[i], w0a[i + 1]),
                             f2fma(f2bc(b), make_float2(w1a[i], w1a[i + 1]), make_float2(b1a[i], b1a[i + 1])));
      float2 om;
      const float2 s = sigm2_pre(u, om);
      const float2 sp = f2mul(om, s);                               // s(1-s)
      const float2 spp = f2fma(f2mul(f2bc(-2.0f), s), sp, sp);      // s'(1-2s)
      s_[k4 + i] = s.x; s_[k4 + i + 1] = s.y;
      sp_[k4 + i] = sp.x; sp_[k4 + i + 1] = sp.y;
      spp_[k4 + i] = spp.x; spp_[k4 + i + 1] = spp.y;
    }
  }
  {
    const uint32_t t0 = c.tlane + cb;
    tc_st_split16<true>(t0 + F_S_HI, t0 + F_S_LO, s_);
    tc_st_split16<true>(t0 + F_SP_HI, t0 + F_SP_LO, sp_);
    tc_st_split16<true>(t0 + F_SPP_HI, t0 + F_SPP_LO, spp_);
  }
  TL(1);
  tc_role_sync(c);
  TL(2);
  // (One issuing warp per role.  Letting three warps issue six MMAs each - one accumulator region per warp, four commits on
  // the role's mbarrier - gives the same bits and a 0.9 % SLOWER step (0.11294 vs 0.11196 ms, profiles/r02_t_ab_issue.log),
  // although the single issuer runs ~350 cycles behind its peers in the timeline.)
  if (c.issuer && elect_one()) {
    tc_fence_after();
    const uint32_t d = c.tbase + cb;
    const uint32_t bs = c.wts_saddr + (uint32_t)offsetof(Wts, BS), bsp = c.wts_saddr + (uint32_t)offsetof(Wts, BSP);
    const uint32_t bspp = c.wts_saddr + (uint32_t)offsetof(Wts, BSPP);
#pragma unroll
    for (uint32_t ks = 0; ks < 2; ks++) {
      // one K step = 8 values = two 16-byte chunks = 2*LBO = 32*N bytes
      tc_mma3(d + F_V0, d + F_S_HI + 8 * ks, d + F_S_LO + 8 * ks, bs + ks * 32 * 16, bs + 4 * NH * NH + ks * 32 * 16, 16,
              tc_idesc(16), ks == 0);
      tc_mma3(d + F_V12, d + F_SP_HI + 8 * ks, d + F_SP_LO + 8 * ks, bsp + ks * 32 * 32, bsp + 4 * 2 * NH * NH + ks * 32 * 32,
              32, tc_idesc(32), ks == 0);
      tc_mma3(d + F_P, d + F_SPP_HI + 8 * ks, d + F_SPP_LO + 8 * ks, bspp + ks * 32 * 48,
              bspp + 4 * 3 * NH * NH + ks * 32 * 48, 48, tc_idesc(48), ks == 0);
    }
    tc_commit(c.mbar);
  }
  __syncwarp();
  if (STASH) {
    // while the tensor pipe works: the 4-channel h of the weight-gradient contraction and of the reverse sweep
#pragma unroll
    for (int k4 = 0; k4 < NH; k4 += 4) {
      const float4 w0v = LD4(&w.w0[k4]), w1v = LD4(&w.w1[k4]);
      const float w0a[4] = {w0v.x, w0v.y, w0v.z, w0v.w}, w1a[4] = {w1v.x, w1v.y, w1v.z, w1v.w};
      const float4 q00 = LD4(&w.ww00[k4]), q01 = LD4(&w.ww01[k4]), q11 = LD4(&w.ww11[k4]);
      const float q00a[4] = {q00.x, q00.y, q00.z, q00.w}, q01a[4] = {q01.x, q01.y, q01.z, q01.w};
      const float q11a[4] = {q11.x, q11.y, q11.z, q11.w};
      float h1[4], h2[4], h3[4];
#pragma unroll
      for (int i = 0; i < 4; i += 2) {
        const float2 w0 = make_float2(w0a[i], w0a[i + 1]), w1 = make_float2(w1a[i], w1a[i + 1]);
        const float2 sp = make_float2(sp_[k4 + i], sp_[k4 + i + 1]), spp = make_float2(spp_[k4 + i], spp_[k4 + i + 1]);
        const float2 d1 = f2fma(f2bc(al1), w0, f2mul(f2bc(al2), w1));
        const float2 q = f2fma(f2bc(al11), make_float2(q00a[i], q00a[i + 1]),
                               f2fma(f2bc(al12), make_float2(q01a[i], q01a[i + 1]), f2mul(f2bc(al22), make_float2(q11a[i], q11a[i + 1]))));
        const float2 a1 = f2mul(sp, w0), a2 = f2mul(sp, w1), a3 = f2fma(sp, d1, f2mul(spp, q));
        h1[i] = a1.x; h1[i + 1] = a1.y; h2[i] = a2.x; h2[i + 1] = a2.y; h3[i] = a3.x; h3[i + 1] = a3.y;
      }
      ST4(&Hrow[(0 * NH + k4) ^ sx], s_[k4], s_[k4 + 1], s_[k4 + 2], s_[k4 + 3]);
      ST4(&Hrow[(1 * NH + k4) ^ sx], h1[0], h1[1], h1[2], h1[3]);
      ST4(&Hrow[(2 * NH + k4) ^ sx], h2[0], h2[1], h2[2], h2[3]);
      ST4(&Hrow[(3 * NH + k4) ^ sx], h3[0], h3[1], h3[2], h3[3]);
    }
  }
  TL(4);
  tc_wait_mma(c);
  TL(3);

  float accN = 0.0f, accD = 0.0f;
#pragma unroll
  for (int j8 = 0; j8 < NH; j8 += 8) {
    float V0[8], V1[8], V2[8], P00[8], P01[8], P11[8];
    const uint32_t t0 = c.tlane + cb;
    tc_ld8(t0 + F_V0 + j8, V0);
    tc_ld8(t0 + F_V12 + j8, V1);
    tc_ld8(t0 + F_V12 + NH + j8, V2);
    tc_ld8(t0 + F_P + j8, P00);
    tc_ld8(t0 + F_P + NH + j8, P01);
    tc_ld8(t0 + F_P + 2 * NH + j8, P11);
    tc_wait_ld(V0); tc_wait_ld(V1); tc_wait_ld(V2); tc_wait_ld(P00); tc_wait_ld(P01); tc_wait_ld(P11);
#pragma unroll
    for (int j4 = 0; j4 < 8; j4 += 4) {
      const float4 b2v = LD4(&w.b2s[j8 + j4]), wov = LD4(&w.wo[j8 + j4]);
      const float b2a[4] = {b2v.x, b2v.y, b2v.z, b2v.w}, woa[4] = {wov.x, wov.y, wov.z, wov.w};
#pragma unroll
      for (int i = 0; i < 4; i += 2) {  // two hidden units per instruction; the sigmoid (MUFU) stays scalar
        const int j = j4 + i;
        const float2 v1 = make_float2(V1[j], V1[j + 1]), v2 = make_float2(V2[j], V2[j + 1]);
        const float2 v3 = f2fma(f2bc(al1), v1, f2fma(f2bc(al2), v2,
                          f2fma(f2bc(al11), make_float2(P00[j], P00[j + 1]),
                                f2fma(f2bc(al12), make_float2(P01[j], P01[j + 1]), f2mul(f2bc(al22), make_float2(P11[j], P11[j + 1]))))));
        float2 om;
        const float2 t = sigm2_pre(f2fma(make_float2(V0[j], V0[j + 1]), f2bc(NEG_LOG2E), make_float2(b2a[i], b2a[i + 1])), om);
        const float2 tp = f2mul(om, t);
        const float2 tpp = f2fma(f2mul(f2bc(-2.0f), t), tp, tp);
        const float2 Q = quad_form2(al11, al12, al22, v1, v2);
        const float2 gD = f2fma(tp, v3, f2mul(tpp, Q));
        // (sequential scalar accumulation: N of the boundary points is one fixed rounding pattern - DESIGN.md section 4 -
        // and this order is the measured one)
        accN = fmaf(woa[i], t.x, accN); accN = fmaf(woa[i + 1], t.y, accN);
        accD = fmaf(woa[i], gD.x, accD); accD = fmaf(woa[i + 1], gD.y, accD);
        if (STASH) {
          // Everything the reverse sweep needs from this unit that does not depend on its seeds (lamN, lamD arrive after
          // the mid-tile exchange), pre-multiplied with wo: the sweep is then 7 packed operations per pair instead of 29,
          // and the six values go back IN PLACE into the tensor-memory columns V0,V1,V2,P00,P01,P11 were just read from
          // (dead until the reverse MMA) - no shared-memory round trip (19 % fewer shared-memory wavefronts).
          // v14: on its own this shortened the MLP roles' tile and the step by 0.3-0.5 % only - the E-net role was within
          // ~300 cycles of the critical path (profiles/r02_ae_*) - and the packed E-net arithmetic on its own made the step
          // 2 % slower; together they take 2.9 % off the step (profiles/r02_ag_*, r02_ai_*).  DESIGN.md section 9.
          const float2 wo2 = make_float2(woa[i], woa[i + 1]);
          const float2 tppp = f2mul(tp, f2fma(f2bc(-6.0f), tp, f2bc(1.0f)));
          const float2 Aq = f2mul(wo2, tp), Bq = f2mul(wo2, tpp);
          const float2 B1 = f2mul(Bq, f2fma(f2bc(2.0f * al11), v1, f2mul(f2bc(al12), v2)));
          const float2 B2 = f2mul(Bq, f2fma(f2bc(al12), v1, f2mul(f2bc(2.0f * al22), v2)));
          const float2 Cq = f2mul(wo2, f2fma(tpp, v3, f2mul(tppp, Q)));
          V0[j] = t.x; V0[j + 1] = t.y; V1[j] = Aq.x; V1[j + 1] = Aq.y; V2[j] = B1.x; V2[j + 1] = B1.y;
          P00[j] = B2.x; P00[j + 1] = B2.y; P01[j] = Cq.x; P01[j + 1] = Cq.y; P11[j] = gD.x; P11[j + 1] = gD.y;
        }
      }
    }
    if (STASH) {
      tc_st8f(t0 + F_V0 + j8, V0);
      tc_st8f(t0 + F_V12 + j8, V1);
      tc_st8f(t0 + F_V12 + NH + j8, V2);
      tc_st8f(t0 + F_P + j8, P00);
      tc_st8f(t0 + F_P + NH + j8, P01);
      tc_st8f(t0 + F_P + 2 * NH + j8, P11);
    }
  }
  Nv = accN;
  Dv = accD;
}

// persistent per-lane accumulators of a warp; one layout for both roles so that the registers are shared
//   MLP warp  : c[0][nt] = mma.sync C fragments of dW2 (16x16), nt = 0,1
//               s0: lane<16 db2[lane] | dwo[lane-16];  s1: lane<16 dW1[lane][0] | dW1[lane-16][1];
//               s2: lane<16 db1[lane] | extra[lane-16] (loss sums, role 0)
//   E-net warp: c[mt][nt] = C fragments of dWE2 (32x32);
//               s0..s4 = dwE[lane], dbE2[lane], dWE1[lane], dbE1[lane], {dWgL,dbgL,dwg,dbg,dbE}[lane]
// The vector sums are packed pairs (colsum2): lane = 16 * half + pair holds, for the two columns 2 pair, 2 pair + 1 of the
// 32-column window of s_k, the sum over the rows of its half; the halves are added in the final fold.
struct TcAcc {
  float c[2][4][4];
  float2 s0, s1, s2, s3, s4;
};
__device__ __forceinline__ void acc2(float2& a, const float2 v) { a = __fadd2_rn(a, v); }
using TcMlpAcc = TcAcc;
using TcEnetAcc = TcAcc;

// Reverse sweep of one MLP evaluation (oracle/closed_form.py:mlp_bwd) for the seeds lamN, lamD
__device__ __forceinline__ void tc_mlp_backward(const Wts& w, TcCtx& c, uint32_t cb, float a, float b, float al1, float al2,
                                                float al11, float al12, float al22, float lamN, float lamD,
                                                float* __restrict__ Hs, float* __restrict__ Gs, int lane,
                                                const float (&extra)[8], TcMlpAcc& acc) {
  const int sx = swz_tc(lane);
  float* Hrow = Hs + lane * ROWH;
  float* Grow = Gs + lane * ROWH;
  float dwo[NH];
  {
    // the forward left {t, wo tp, wo tpp (2 al11 v1 + al12 v2), wo tpp (al12 v1 + 2 al22 v2), wo (tpp v3 + tppp Q), gD} of every
    // hidden unit in the tensor-memory columns of V0,V1,V2,P00,P01,P11; with the seeds known the adjoints are
    //   vbar0 = lamN A + lamD C, vbar1 = lamD B1, vbar2 = lamD B2, vbar3 = lamD A, dwo = lamN t + lamD gD.
    // Eight units at a time: all six loads of a block precede its stores (vbar lo of channels 2, 3 lands on the block's
    // own t / A columns), and a block's vbar goes to tensor memory and to the stash at once - nothing stays in registers.
    const uint32_t t0 = c.tlane + cb;
    tc_wait_st();  // the forward's parking stores (long complete by now; the wait makes the order explicit)
#pragma unroll
    for (int j8 = 0; j8 < NH; j8 += 8) {
      float T[8], A[8], B1[8], B2[8], C[8], GD[8];
      tc_ld8(t0 + F_V0 + j8, T);
      tc_ld8(t0 + F_V12 + j8, A);
      tc_ld8(t0 + F_V12 + NH + j8, B1);
      tc_ld8(t0 + F_P + j8, B2);
      tc_ld8(t0 + F_P + NH + j8, C);
      tc_ld8(t0 + F_P + 2 * NH + j8, GD);
      tc_wait_ld(T); tc_wait_ld(A); tc_wait_ld(B1); tc_wait_ld(B2); tc_wait_ld(C); tc_wait_ld(GD);
      float vb[4][8];
#pragma unroll
      for (int i = 0; i < 8; i += 2) {
        const float2 a2 = make_float2(A[i], A[i + 1]);
        const float2 v0 = f2fma(f2bc(lamN), a2, f2mul(f2bc(lamD), make_float2(C[i], C[i + 1])));
        const float2 v1 = f2mul(f2bc(lamD), make_float2(B1[i], B1[i + 1]));
        const float2 v2 = f2mul(f2bc(lamD), make_float2(B2[i], B2[i + 1]));
        const float2 v3 = f2mul(f2bc(lamD), a2);
        const float2 dw = f2fma(f2bc(lamN), make_float2(T[i], T[i + 1]), f2mul(f2bc(lamD), make_float2(GD[i], GD[i + 1])));
        vb[0][i] = v0.x; vb[0][i + 1] = v0.y; vb[1][i] = v1.x; vb[1][i + 1] = v1.y;
        vb[2][i] = v2.x; vb[2][i + 1] = v2.y; vb[3][i] = v3.x; vb[3][i + 1] = v3.y;
        dwo[j8 + i] = dw.x; dwo[j8 + i + 1] = dw.y;
      }
#pragma unroll
      for (int ch = 0; ch < 4; ch++) {
        ST4(&Grow[(ch * NH + j8) ^ sx], vb[ch][0], vb[ch][1], vb[ch][2], vb[ch][3]);
        ST4(&Grow[(ch * NH + j8 + 4) ^ sx], vb[ch][4], vb[ch][5], vb[ch][6], vb[ch][7]);
        tc_st_split8(t0 + B_VB_HI + ch * NH + j8, t0 + B_VB_LO + ch * NH + j8, vb[ch]);
      }
    }
  }
  TL(7);
  tc_role_sync(c);  // (also orders the stash writes above before the fragment loads below: bar.sync)
  TL(8);
  if (c.issuer && elect_one()) {
    tc_fence_after();
    const uint32_t d = c.tbase + cb;
    const uint32_t bw = c.wts_saddr + (uint32_t)offsetof(Wts, BWT);
#pragma unroll
    for (uint32_t ch = 0; ch < 4; ch++)
#pragma unroll
      for (uint32_t ks = 0; ks < 2; ks++)
        tc_mma3(d + B_HB + ch * NH, d + B_VB_HI + ch * NH + 8 * ks, d + B_VB_LO + ch * NH + 8 * ks, bw + ks * 32 * 16,
                bw + 4 * NH * NH + ks * 32 * 16, 16, tc_idesc(16), ks == 0);
    tc_commit(c.mbar);
  }
  __syncwarp();

  // ---- while the tensor core runs: dW2[j][k] += sum_{p,c} G[p][c][j] * H[p][c][k] (mma.sync, 3xTF32) ----
  {
    // rows po*8 + t and po*8 + t + 4: swz_tc = t << 3 and (t << 3) | 4
    const int g = lane >> 2, t = lane & 3, tx = t << 3, ty = tx | 4;
#pragma unroll 1
    for (int ch = 0; ch < 4; ch++) {
#pragma unroll
      for (int po = 0; po < 4; po++) {
        const float* Ga = Gs + (po * 8 + t) * ROWH;
        const float* Gb = Ga + 4 * ROWH;
        const float* Ha = Hs + (po * 8 + t) * ROWH;
        const float* Hb = Ha + 4 * ROWH;
        const int ca = (ch * NH + g) ^ tx, cbb = (ch * NH + g + 8) ^ tx;
        const int da = (ch * NH + g) ^ ty, dbb = (ch * NH + g + 8) ^ ty;
        uint32_t ah[4], al[4];
        split_tf32(Ga[ca], ah[0], al[0]);
        split_tf32(Ga[cbb], ah[1], al[1]);
        split_tf32(Gb[da], ah[2], al[2]);
        split_tf32(Gb[dbb], ah[3], al[3]);
        uint32_t bh0, bl0, bh1, bl1;
        split_tf32(Ha[ca], bh0, bl0);
        split_tf32(Hb[da], bh1, bl1);
        // even / odd k-steps accumulate into separate fragments: four independent HMMA chains instead of two (the
        // phase is bound by the accumulate latency of the legacy tensor path, not by its throughput)
        mma_3xtf32(acc.c[po & 1][0], ah, al, bh0, bh1, bl0, bl1);
        split_tf32(Ha[cbb], bh0, bl0);
        split_tf32(Hb[dbb], bh1, bl1);
        mma_3xtf32(acc.c[po & 1][1], ah, al, bh0, bh1, bl0, bl1);
      }
    }
  }
  __syncwarp();  // all fragment loads done: channel 1..3 regions of the stash rows may be reused
  // ---- db2 (= column sums of vbar channel 0) and dwo ----
#pragma unroll
  for (int j4 = 0; j4 < NH; j4 += 4) ST4(&Grow[(NH + j4) ^ sx], dwo[j4], dwo[j4 + 1], dwo[j4 + 2], dwo[j4 + 3]);
  __syncwarp();
  TL(9);
  // (Handing these column sums to the group's E-net warp - it has finished its own tile by then - keeps the bits and makes the
  // step 0.9 % SLOWER, 0.11338 vs 0.11233 ms, profiles/r02_v_ab_colsum_handoff.log: after the geometry hand-off the E-net
  // role has no slack left to give.)
  acc2(acc.s0, colsum2<ROWH>(Gs, 2 * (lane & 15), lane >> 4));

  // ---- hbar = W2^T vbar is in TMEM now: layer-1 reverse sweep ----
  TL(10);
  tc_wait_mma(c);
  TL(11);
#pragma unroll
  for (int k8 = 0; k8 < NH; k8 += 8) {
    float hb0[8], hb1[8], hb2[8], hb3[8];
    const uint32_t t0 = c.tlane + cb + B_HB;
    tc_ld8(t0 + 0 * NH + k8, hb0);
    tc_ld8(t0 + 1 * NH + k8, hb1);
    tc_ld8(t0 + 2 * NH + k8, hb2);
    tc_ld8(t0 + 3 * NH + k8, hb3);
    tc_wait_ld(hb0); tc_wait_ld(hb1); tc_wait_ld(hb2); tc_wait_ld(hb3);
#pragma unroll
    for (int k4 = 0; k4 < 8; k4 += 4) {
      const int kk = k8 + k4;
      const float4 sv = LD4(&Hrow[kk ^ sx]);  // h channel 0 = s_k
      const float sa[4] = {sv.x, sv.y, sv.z, sv.w};
      float spa[4];
      {  // s(1-s) with 1 - s from the exponential of the forward's pre-activation (same expression, same bits), not from s
        const float4 w0sv = LD4(&w.w0s[kk]), w1sv = LD4(&w.w1s[kk]), b1sv = LD4(&w.b1s[kk]);
        const float w0sa[4] = {w0sv.x, w0sv.y, w0sv.z, w0sv.w}, w1sa[4] = {w1sv.x, w1sv.y, w1sv.z, w1sv.w};
        const float b1sa[4] = {b1sv.x, b1sv.y, b1sv.z, b1sv.w};
#pragma unroll
        for (int i = 0; i < 4; i += 2) {
          const float2 s = make_float2(sa[i], sa[i + 1]);
          const float2 u = f2fma(f2bc(a), make_float2(w0sa[i], w0sa[i + 1]),
                                 f2fma(f2bc(b), make_float2(w1sa[i], w1sa[i + 1]), make_float2(b1sa[i], b1sa[i + 1])));
          const float2 sp = f2mul(one_minus_sigm2_pre(u, s), s);
          spa[i] = sp.x; spa[i + 1] = sp.y;
        }
      }
      const float4 w0v = LD4(&w.w0[kk]), w1v = LD4(&w.w1[kk]);
      const float4 q00 = LD4(&w.ww00[kk]), q01 = LD4(&w.ww01[kk]), q11 = LD4(&w.ww11[kk]);
      const float w0a[4] = {w0v.x, w0v.y, w0v.z, w0v.w}, w1a[4] = {w1v.x, w1v.y, w1v.z, w1v.w};
      const float q00a[4] = {q00.x, q00.y, q00.z, q00.w}, q01a[4] = {q01.x, q01.y, q01.z, q01.w};
      const float q11a[4] = {q11.x, q11.y, q11.z, q11.w};
      float o0[4], o1[4], ob[4];
      // two hidden units per instruction (packed FFMA2 / FMUL2): same operations, same rounding, half the issue slots
#pragma unroll
      for (int i = 0; i < 4; i += 2) {
        const float2 h0 = make_float2(hb0[k4 + i], hb0[k4 + i + 1]), h1 = make_float2(hb1[k4 + i], hb1[k4 + i + 1]);
        const float2 h2 = make_float2(hb2[k4 + i], hb2[k4 + i + 1]), h3 = make_float2(hb3[k4 + i], hb3[k4 + i + 1]);
        const float2 s = make_float2(sa[i], sa[i + 1]);
        const float2 w0 = make_float2(w0a[i], w0a[i + 1]), w1 = make_float2(w1a[i], w1a[i + 1]);
        const float2 q00p = make_float2(q00a[i], q00a[i + 1]), q01p = make_float2(q01a[i], q01a[i + 1]);
        const float2 q11p = make_float2(q11a[i], q11a[i + 1]);
        const float2 sp = make_float2(spa[i], spa[i + 1]);
        const float2 spp = f2fma(f2mul(f2bc(-2.0f), s), sp, sp);
        const float2 sppp = f2mul(sp, f2fma(f2bc(-6.0f), sp, f2bc(1.0f)));
        const float2 d1 = f2fma(f2bc(al1), w0, f2mul(f2bc(al2), w1));
        const float2 q = f2fma(f2bc(al11), q00p, f2fma(f2bc(al12), q01p, f2mul(f2bc(al22), q11p)));
        const float2 ubar = f2fma(h0, sp, f2fma(f2fma(h1, w0, f2fma(h2, w1, f2mul(h3, d1))), spp, f2mul(f2mul(h3, q), sppp)));
        const float2 r0 = f2fma(h1, sp, f2fma(h3, f2fma(sp, f2bc(al1), f2mul(spp, f2fma(f2bc(2.0f * al11), w0, f2mul(f2bc(al12), w1)))),
                                         f2mul(ubar, f2bc(a))));
        const float2 r1 = f2fma(h2, sp, f2fma(h3, f2fma(sp, f2bc(al2), f2mul(spp, f2fma(f2bc(al12), w0, f2mul(f2bc(2.0f * al22), w1)))),
                                         f2mul(ubar, f2bc(b))));
        o0[i] = r0.x; o0[i + 1] = r0.y;
        o1[i] = r1.x; o1[i + 1] = r1.y;
        ob[i] = ubar.x; ob[i + 1] = ubar.y;
      }
      ST4(&Hrow[(1 * NH + kk) ^ sx], o0[0], o0[1], o0[2], o0[3]);
      ST4(&Hrow[(2 * NH + kk) ^ sx], o1[0], o1[1], o1[2], o1[3]);
      ST4(&Hrow[(3 * NH + kk) ^ sx], ob[0], ob[1], ob[2], ob[3]);
    }
  }
  ST4(&Hrow[0 ^ sx], extra[0], extra[1], extra[2], extra[3]);
  ST4(&Hrow[4 ^ sx], extra[4], extra[5], extra[6], extra[7]);
  __syncwarp();
  TL(12);
  acc2(acc.s1, colsum2<ROWH>(Hs, NH + 2 * (lane & 15), lane >> 4));               // columns 16..47: dw0 | dw1
  acc2(acc.s2, colsum2<ROWH>(Hs, (3 * NH + 2 * (lane & 15)) & 63, lane >> 4));    // columns 48..63: db1 ; 0..15: extras
  __syncwarp();
}

// loss sums only (fine-tune mode: no base-MLP reverse sweep); role 0
__device__ __forceinline__ void tc_mlp_extras_only(float* __restrict__ Hs, int lane, const float (&extra)[8], TcMlpAcc& acc) {
  const int sx = swz_tc(lane);
  float* Hrow = Hs + lane * ROWH;
  __syncwarp();
  ST4(&Hrow[0 ^ sx], extra[0], extra[1], extra[2], extra[3]);
  ST4(&Hrow[4 ^ sx], extra[4], extra[5], extra[6], extra[7]);
  __syncwarp();
  const float2 v = colsum2<ROWH>(Hs, (3 * NH + 2 * (lane & 15)) & 63, lane >> 4);  // same window as in tc_mlp_backward
  if ((lane & 15) >= 8 && (lane & 15) < 12) acc2(acc.s2, v);                       // its columns 0..7: the extras
  __syncwarp();
}

// ---------------------------------------------------------------------------------------------
// E(R) network (poc/main.py:249-253; train.py:50-52) and gate (poc/main.py:262-264; train.py:48-49)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float tc_gate_forward(const Wts& w, float R);
template <bool STASH>
__device__ __forceinline__ float tc_enet_forward(const Wts& w, TcCtx& c, float R, float* __restrict__ E1row,
                                                 float* __restrict__ Vrow, int sx, float& gate_out) {
  const uint32_t t0 = c.tlane + TC_E_BASE;
#pragma unroll
  for (int k16 = 0; k16 < NE; k16 += 16) {
    float e1[16];
#pragma unroll
    for (int k4 = 0; k4 < 16; k4 += 4) {
      // pre-activations arrive as the MUFU.EX2 argument (weights pre-multiplied by -log2 e): one rounding in front of the
      // exponential instead of two, like the MLP roles
      const float4 wv = LD4(&w.WE1s[k16 + k4]), bv = LD4(&w.bE1s[k16 + k4]);
      // two units per instruction (FFMA2 / FADD2), the same operations and roundings as the scalar form
      float2 oa, ob;
      const float2 sa = sigm2_pre(f2fma(f2bc(R), make_float2(wv.x, wv.y), make_float2(bv.x, bv.y)), oa);
      const float2 sb = sigm2_pre(f2fma(f2bc(R), make_float2(wv.z, wv.w), make_float2(bv.z, bv.w)), ob);
      e1[k4 + 0] = sa.x; e1[k4 + 1] = sa.y; e1[k4 + 2] = sb.x; e1[k4 + 3] = sb.y;
      if (STASH) {  // s'(1-s) for the reverse sweep: the stash keeps e1 only
        const float2 pa = f2mul(oa, sa), pb = f2mul(ob, sb);
        tc_st4f(c.tlane + TC_SP_PARK + k16 + k4, pa.x, pa.y, pb.x, pb.y);
      }
      if (STASH) ST4(&E1row[(k16 + k4) ^ sx], e1[k4], e1[k4 + 1], e1[k4 + 2], e1[k4 + 3]);
    }
    tc_st_split16<true>(t0 + E_A_HI + k16, t0 + E_A_LO + k16, e1);
  }
  TL(1);
  tc_role_sync(c);
  TL(2);
  if (c.issuer && elect_one()) {
    tc_fence_after();
    const uint32_t d = c.tbase + TC_E_BASE;
    const uint32_t be = c.wts_saddr + (uint32_t)offsetof(Wts, BE);
#pragma unroll
    for (uint32_t ks = 0; ks < 4; ks++)
      tc_mma3(d + E_D, d + E_A_HI + 8 * ks, d + E_A_LO + 8 * ks, be + ks * 32 * 32, be + 4 * NE * NE + ks * 32 * 32, 32,
              tc_idesc(32), ks == 0);
    tc_commit(c.mbar);
  }
  __syncwarp();
  // the gate (ten sigmoids of R, independent of the MMA) while the tensor core runs: this role has no stash writes to hide
  // its forward MMAs behind (-0.2 %, same bits, profiles/r02_ay_*; moving the e1 stash writes here as well keeps 32 more
  // values live across the barrier and is 1.6 % slower, r02_ax_*)
  gate_out = tc_gate_forward(w, R);
  tc_wait_mma(c);
  TL(3);
  float E = w.bE;
#pragma unroll
  for (int j16 = 0; j16 < NE; j16 += 16) {
    float v[16];
    tc_ld16(t0 + E_D + j16, v);
    tc_wait_ld(v);
#pragma unroll
    for (int j4 = 0; j4 < 16; j4 += 4) {
      const float4 b2v = LD4(&w.bE2s[j16 + j4]), wEv = LD4(&w.wE[j16 + j4]);
      const float b2a[4] = {b2v.x, b2v.y, b2v.z, b2v.w}, wEa[4] = {wEv.x, wEv.y, wEv.z, wEv.w};
      float e2[4];
#pragma unroll
      for (int i = 0; i < 4; i += 2) {
        float2 om;
        const float2 s2 = sigm2_pre(f2fma(make_float2(v[j4 + i], v[j4 + i + 1]), f2bc(NEG_LOG2E), make_float2(b2a[i], b2a[i + 1])), om);
        if (STASH) {  // v is consumed: its registers take s'(1-s) for the reverse sweep
          const float2 sp = f2mul(om, s2);
          v[j4 + i] = sp.x; v[j4 + i + 1] = sp.y;
        }
        e2[i] = s2.x; e2[i + 1] = s2.y;
        E = fmaf(wEa[i], e2[i], E);
        E = fmaf(wEa[i + 1], e2[i + 1], E);
      }
      if (STASH) ST4(&Vrow[(j16 + j4) ^ sx], e2[0], e2[1], e2[2], e2[3]);
    }
    if (STASH) tc_st16f(t0 + E_D + j16, v);  // D is dead until the reverse MMA; the stash keeps e2 only
  }
  return E;
}

__device__ __forceinline__ float tc_gate_forward(const Wts& w, float R) {
  float g = w.bg;
#pragma unroll
  for (int i = 0; i < NL; i += 2) {
    const float2 s2 = sigm2_pre(f2fma(f2bc(R), make_float2(w.WgLs[i], w.WgLs[i + 1]), make_float2(w.bgLs[i], w.bgLs[i + 1])));
    g = fmaf(w.wg[i], s2.x, g);
    g = fmaf(w.wg[i + 1], s2.y, g);
  }
  return g;
}

__device__ __forceinline__ void tc_enet_backward(const Wts& w, TcCtx& c, float R, float Ebar, float gbar, bool gate_grads,
                                                 float* __restrict__ E1s, float* __restrict__ Vs, int lane, TcEnetAcc& acc) {
  const int sx = swz_tc(lane);
  float* E1row = E1s + lane * ROWE;
  float* Vrow = Vs + lane * ROWE;
  const uint32_t t0 = c.tlane + TC_E_BASE;
  tc_wait_st();  // the forward's s'(1-s) stores (D, TC_SP_PARK)
  __syncwarp();
  // ---- dwE[j] = sum_p Ebar_p e2[p][j] (Vs still holds e2) ----
  {
    float2 plain, weighted;
    colsum2_w<ROWE>(Vs, 2 * (lane & 15), lane >> 4, Ebar, plain, weighted);
    acc2(acc.s0, weighted);
  }
  __syncwarp();
#pragma unroll
  for (int j16 = 0; j16 < NE; j16 += 16) {
    float vbar[16], sp[16];
    tc_ld16(t0 + E_D + j16, sp);  // s'(1-s) of layer 2 as the forward formed it (1 - s = e s); D is written next by the
    tc_wait_ld(sp);               // reverse MMA below
#pragma unroll
    for (int j4 = 0; j4 < 16; j4 += 4) {
      const float4 wEv = LD4(&w.wE[j16 + j4]);
      const float wEa[4] = {wEv.x, wEv.y, wEv.z, wEv.w};
#pragma unroll
      for (int i = 0; i < 4; i += 2) {
        const float2 vb = f2mul(f2mul(f2bc(Ebar), make_float2(wEa[i], wEa[i + 1])), make_float2(sp[j4 + i], sp[j4 + i + 1]));
        vbar[j4 + i] = vb.x; vbar[j4 + i + 1] = vb.y;
      }
      ST4(&Vrow[(j16 + j4) ^ sx], vbar[j4], vbar[j4 + 1], vbar[j4 + 2], vbar[j4 + 3]);
    }
    tc_st_split16<false>(t0 + E_A_HI + j16, t0 + E_A_LO + j16, vbar);
  }
  TL(7);
  tc_role_sync(c);
  TL(8);
  if (c.issuer && elect_one()) {
    tc_fence_after();
    const uint32_t d = c.tbase + TC_E_BASE;
    const uint32_t be = c.wts_saddr + (uint32_t)offsetof(Wts, BET);
#pragma unroll
    for (uint32_t ks = 0; ks < 4; ks++)
      tc_mma3(d + E_D, d + E_A_HI + 8 * ks, d + E_A_LO + 8 * ks, be + ks * 32 * 32, be + 4 * NE * NE + ks * 32 * 32, 32,
              tc_idesc(32), ks == 0);
    tc_commit(c.mbar);
  }
  __syncwarp();
  // ---- while the tensor core runs: dWE2[j][k] += sum_p V[p][j] * E1[p][k] (mma.sync, 3xTF32) ----
  {
    const int g = lane >> 2, t = lane & 3, tx = t << 3, ty = tx | 4;  // swz_tc of rows ks*8 + t and ks*8 + t + 4
#pragma unroll 1
    for (int ks = 0; ks < 4; ks++) {
      const float* Va = Vs + (ks * 8 + t) * ROWE;
      const float* Vb = Va + 4 * ROWE;
      const float* Ea = E1s + (ks * 8 + t) * ROWE;
      const float* Eb = Ea + 4 * ROWE;
      uint32_t ah[2][4], al[2][4];
#pragma unroll
      for (int mt = 0; mt < 2; mt++) {
        split_tf32(Va[(mt * 16 + g) ^ tx], ah[mt][0], al[mt][0]);
        split_tf32(Va[(mt * 16 + g + 8) ^ tx], ah[mt][1], al[mt][1]);
        split_tf32(Vb[(mt * 16 + g) ^ ty], ah[mt][2], al[mt][2]);
        split_tf32(Vb[(mt * 16 + g + 8) ^ ty], ah[mt][3], al[mt][3]);
      }
#pragma unroll
      for (int nt = 0; nt < 4; nt++) {
        uint32_t bh0, bl0, bh1, bl1;
        split_tf32(Ea[(nt * 8 + g) ^ tx], bh0, bl0);
        split_tf32(Eb[(nt * 8 + g) ^ ty], bh1, bl1);
        mma_3xtf32(acc.c[0][nt], ah[0], al[0], bh0, bh1, bl0, bl1);
        mma_3xtf32(acc.c[1][nt], ah[1], al[1], bh0, bh1, bl0, bl1);
      }
    }
  }
  TL(9);
  acc2(acc.s1, colsum2<ROWE>(Vs, 2 * (lane & 15), lane >> 4));  // dbE2
  __syncwarp();                      // Vs rows may now be overwritten
  // ---- e1bar = WE2^T vbar is in TMEM: layer-1 reverse sweep; ubar_k -> Vs row ----
  TL(10);
  tc_wait_mma(c);
  TL(11);
#pragma unroll
  for (int k16 = 0; k16 < NE; k16 += 16) {
    float eb[16], sp1[16];
    tc_ld16(t0 + E_D + k16, eb);
    tc_ld16(c.tlane + TC_SP_PARK + k16, sp1);  // s'(1-s) of layer 1 as the forward formed it (1 - s = e s)
    tc_wait_ld(eb); tc_wait_ld(sp1);
#pragma unroll
    for (int k4 = 0; k4 < 16; k4 += 4) {
      float ub[4];
#pragma unroll
      for (int i = 0; i < 4; i += 2) {
        const float2 u = f2mul(make_float2(eb[k4 + i], eb[k4 + i + 1]), make_float2(sp1[k4 + i], sp1[k4 + i + 1]));
        ub[i] = u.x; ub[i + 1] = u.y;
      }
      ST4(&Vrow[(k16 + k4) ^ sx], ub[0], ub[1], ub[2], ub[3]);
    }
  }
  // ---- gate reverse sweep + dbE -> E1s row (free now) ----
  {
    float ch[32];
#pragma unroll
    for (int i = 0; i < NL; i += 2) {
      float2 om;
      const float2 s2 = sigm2_pre(f2fma(f2bc(R), make_float2(w.WgLs[i], w.WgLs[i + 1]), make_float2(w.bgLs[i], w.bgLs[i + 1])), om);
      const float2 ub = gate_grads ? f2mul(f2mul(f2bc(gbar), make_float2(w.wg[i], w.wg[i + 1])), f2mul(om, s2)) : f2bc(0.0f);
      const float2 ur = f2mul(ub, f2bc(R));
      const float2 gs = gate_grads ? f2mul(f2bc(gbar), s2) : f2bc(0.0f);
      ch[i] = ur.x; ch[i + 1] = ur.y;
      ch[10 + i] = ub.x; ch[10 + i + 1] = ub.y;
      ch[20 + i] = gs.x; ch[20 + i + 1] = gs.y;
    }
    ch[30] = gate_grads ? gbar : 0.0f;
    ch[31] = Ebar;
#pragma unroll
    for (int c4 = 0; c4 < 32; c4 += 4) ST4(&E1row[c4 ^ sx], ch[c4], ch[c4 + 1], ch[c4 + 2], ch[c4 + 3]);
  }
  __syncwarp();
  {
    float2 plain, weighted;
    colsum2_w<ROWE>(Vs, 2 * (lane & 15), lane >> 4, R, plain, weighted);
    acc2(acc.s2, weighted);  // dWE1[k] = sum_p ubar_k R_p
    acc2(acc.s3, plain);     // dbE1
  }
  acc2(acc.s4, colsum2<ROWE>(E1s, 2 * (lane & 15), lane >> 4));
  __syncwarp();
}

// ---------------------------------------------------------------------------------------------
// the fused kernel.  NEV = MLP evaluations per point (2: poc, 1: train.py); TRAIN = with reverse sweep
//   warp = role * 4 + group;  role < NEV: MLP evaluation, role == NEV: E-net + gate
// ---------------------------------------------------------------------------------------------
// final fold of a packed vector sum: add the two row halves (lanes l and l + 16), lanes 0..15 store their two columns
template <typename EntryOf>
__device__ __forceinline__ void fold_pair(float* __restrict__ myrow, float2 v, int lane, EntryOf entry_of) {
  v.x += __shfl_xor_sync(0xffffffffu, v.x, 16);
  v.y += __shfl_xor_sync(0xffffffffu, v.y, 16);
  if (lane < 16) {
    const int a = entry_of(2 * lane), b = entry_of(2 * lane + 1);
    if (a >= 0) myrow[a] = v.x;
    if (b >= 0) myrow[b] = v.y;
  }
}

// Kernel parameters: the launch description; the INLINE instantiations (the *_host entry) also carry theta and the loss
// weights by value (6 KB of parameter space; sm_100 takes up to 32 KB), so that no host-to-device copy has to precede
// the kernel.
constexpr int TC_REG_MLP = 184, TC_REG_ENET = 136;  // setmaxnreg targets of the poc training kernel (see the kernel's tail)
static_assert(128 * TC_REG_ENET + 256 * TC_REG_MLP <= 384 * 168, "register rebalancing must fit the launch allocation");

struct TcParamsPlain {
  StepParams p;
  double w[4];  // loss weights by value when p.w_by_value
};
struct TcParamsInline {
  StepParams p;
  double w[4];
  alignas(16) float theta[NTHETA + 3];
};

template <int NEV, bool TRAIN, bool INLINE>
__global__ void __launch_bounds__((NEV + 1) * 128, 1)
pinn_step_tc_kernel(const __grid_constant__ typename std::conditional<INLINE, TcParamsInline, TcParamsPlain>::type q) {
  const StepParams& p = q.p;
  constexpr int G = 4;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  Wts& w = *reinterpret_cast<Wts*>(smem_raw);
  uint64_t* mbars = reinterpret_cast<uint64_t*>(smem_raw + sizeof(Wts));  // [0]: weight copy, [1..3]: roles
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem_raw + sizeof(Wts) + 32);
  uint64_t* cfull = reinterpret_cast<uint64_t*>(smem_raw + sizeof(Wts) + 40);  // [COORD_STAGES]: bulk coordinate copies landed
  float2* mbox = reinterpret_cast<float2*>(smem_raw + sizeof(Wts) + 64);
  float* stash = reinterpret_cast<float*>(smem_raw + sizeof(Wts) + 64 + sizeof(float2) * G * 2 * 3 * 32);
  unsigned char* cstage = smem_raw + tc_smem_bytes<NEV>() - COORD_STAGES * COORD_STAGE_BYTES - GEO_BYTES;
  float4* geo = reinterpret_cast<float4*>(smem_raw + tc_smem_bytes<NEV>() - GEO_BYTES);  // [2][128][3]

  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);  // provably warp-uniform: role/group branches and MMA operands
  const int role = warp >> 2, grp = warp & 3;
  const bool is_mlp = role < NEV;
  const int sx = swz_tc(lane);
  TLK(0);
  // CTA 0 times itself (SM cycles and nanoseconds, entry to the end of its tile loop): the effective SM clock of the launch,
  // read back by pinn_step_kernel_clock.  It is lower than the clock nvidia-smi samples while the tensor pipe is in use.
  // (start values parked in two free slots of the 64-byte barrier block, not in registers that would stay live)
  uint32_t* clk0_slot = reinterpret_cast<uint32_t*>(smem_raw + sizeof(Wts) + 36);
  unsigned long long* ns0_slot = reinterpret_cast<unsigned long long*>(smem_raw + sizeof(Wts) + 56);
  if (blockIdx.x == 0 && tid == 0) {
    unsigned long long ns0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns0));
    *ns0_slot = ns0;
    *clk0_slot = (uint32_t)clock();
  }

  // ---- one-time setup: TMEM allocation (warp 0), mbarriers, weight image by TMA bulk copy ----
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (tid == 32) {
#pragma unroll
    for (int i = 0; i < 4; i++) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&mbars[i])));
#pragma unroll
    for (int i = 0; i < COORD_STAGES; i++) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&cfull[i])));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  // launched as a programmatic dependent (launch_pdl): everything above needs no global memory and overlaps the tail of
  // the kernel in front (reduction / Adam / sampler); from here on their results are read
  pdl_wait();
  const int slot = grp * 32 + lane;
  const bool stager = !is_mlp && !p.grid.on;  // the E-net warp (the role with slack) moves its group's coordinates
  // The launches of the *_host entry (INLINE: theta and weights in the kernel parameters, coordinates usually page-locked
  // host memory read in place) move the full super-tiles of 16-byte aligned columns as bulk copies, one issuing thread.
  // Launches on device-resident batches keep the per-lane cp.async stage and carry no bulk code at all: with it the step on
  // HBM-resident inputs measured 1.7 % slower (0.1166 vs 0.1146 ms, tools/ab_time.py on one box, whichever warp issues and
  // whoever waits), against 3 % gained when the coordinates cross PCIe.
  const bool cbulk = INLINE && TRAIN && !p.grid.on &&
                     ((((uintptr_t)p.x | (uintptr_t)p.y | (uintptr_t)p.z | (uintptr_t)p.R | (uintptr_t)p.mask) & 15u) == 0);
  auto tile_bulk = [&](long long st) { return INLINE && cbulk && (st * 128 + 128 <= p.n); };
  const bool bulk_issuer = stager && grp == 0 && lane == 0;  // in the warp that SYNCS on the E-net role barrier (see below)
  if (stager && tile_bulk(blockIdx.x)) {
    if (bulk_issuer) coord_stage_issue_bulk(p, cstage, &cfull[0], blockIdx.x);
  } else if (stager) {
    const long long i0 = (long long)blockIdx.x * 128 + slot;
    coord_stage_issue(p, cstage, slot, i0 < p.n ? i0 : p.n - 1);
    cp_async_commit();
  }

  // ---- weights: theta arrives in shared memory by ONE TMA bulk copy (6080 of its 6084 bytes; bulk copies move multiples
  //      of 16 bytes), every thread then takes part in turning it into the image the kernel reads: layer-1 rows, the
  //      pre-multiplied and hi/lo-split tensor-core operands in the canonical K-major layout.  No separate prep launch.
  {
    float* th_s = stash;  // the stash is free until the first super-tile
    constexpr uint32_t TH_BULK = (NTHETA * 4 / 16) * 16;
    const bool bulk_ok = ((uintptr_t)p.theta & 15u) == 0;
    if constexpr (INLINE) {
      // theta came with the kernel parameters: warp-uniform 16-byte reads (the constant cache serves one address per
      // request), lanes 0..3 scatter the four values
      const float4* src = reinterpret_cast<const float4*>(q.theta);
      for (int j = warp; j < (NTHETA + 3) / 4; j += (NEV + 1) * 4) {
        const float4 v = src[j];
        const float val = lane == 0 ? v.x : lane == 1 ? v.y : lane == 2 ? v.z : v.w;
        if (lane < 4 && 4 * j + lane < NTHETA) th_s[4 * j + lane] = val;
      }
    } else if (p.theta_from_tensors) {
      // the caller's 16 tensors (float32 / float64, (out,in) or train.py's (in,out) layout): gathered here, converted
      // to float32 like `theta.float()` would
      for (int i = tid; i < NTHETA; i += blockDim.x) {
        int k, off;
        theta_locate(i, k, off);
        int j = i - off;
        if (p.tensors_in_out) j = in_out_index(k, j);
        th_s[i] = p.tensors_f64 ? (float)static_cast<const double*>(p.theta_tensors[k])[j]
                                : static_cast<const float*>(p.theta_tensors[k])[j];
      }
    } else if (bulk_ok) {
      if (tid == 32) {
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(&mbars[0])), "r"(TH_BULK) : "memory");
        asm volatile(
            "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(th_s)),
            "l"(p.theta), "r"(TH_BULK), "r"(smem_u32(&mbars[0]))
            : "memory");
      }
      for (int i = TH_BULK / 4 + tid; i < NTHETA; i += blockDim.x) th_s[i] = p.theta[i];
      mbar_wait(smem_u32(&mbars[0]), 0);
    } else {  // unaligned caller buffer: plain loads
      for (int i = tid; i < NTHETA; i += blockDim.x) th_s[i] = p.theta[i];
    }
    __syncthreads();
    build_weight_image(th_s, &w, tid, blockDim.x);
    // the tensor cores read the operand images through the async proxy
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
  }

  // The rest of the kernel is instantiated once per kind of role, in two disjoint branches: with the role a compile-time
  // constant each branch only contains its own code, and (poc training kernel) the branches start with setmaxnreg so
  // that the two MLP warpgroups take over the registers the E-net warpgroup does not need.
  auto run_role = [&](auto mlp_tag) {
    constexpr bool IS_MLP = decltype(mlp_tag)::value;
    TcCtx c;
    c.tbase = __shfl_sync(0xffffffffu, *tmem_slot, 0);
    c.tlane = c.tbase + ((uint32_t)(grp * 32) << 16);
    c.mbar = smem_u32(&mbars[1 + role]);
    c.phase = 0;
    c.bar_id = 5 + role;
    c.issuer = (grp == 0);
    c.wts_saddr = smem_u32(&w);
    const uint32_t cb = IS_MLP ? (uint32_t)role * TC_MLP_COLS : TC_E_BASE;

    float* gstash = stash + grp * tc_group_stash_floats<NEV>();
    float* Hs = gstash + (IS_MLP ? role * EVAL_STASH : NEV * EVAL_STASH);
    float* Gs = Hs + (IS_MLP ? 32 * ROWH : 32 * ROWE);  // for the E-net warp: Hs = E1s, Gs = Vs
    float2* gbox = mbox + grp * (2 * 3 * 32);

    double wpde = 0.0, wbc1 = 0.0, wbc2 = 0.0;
    if (TRAIN) {
      if (INLINE || p.w_by_value) { wpde = q.w[0]; wbc1 = q.w[1]; wbc2 = q.w[2]; }
      else { wpde = p.weights[0]; wbc1 = p.weights[1]; wbc2 = p.weights[2]; }
    }
    const float w_pde = (float)wpde, w_bc1 = (float)wbc1, w_bc2 = (float)wbc2;
    const float sN = p.vc.sN, cL = p.vc.cL, cV = p.vc.cV, cE = p.vc.cE;

    TcAcc acc;
  #pragma unroll
    for (int a = 0; a < 2; a++)
  #pragma unroll
      for (int b = 0; b < 4; b++)
  #pragma unroll
        for (int cc = 0; cc < 4; cc++) acc.c[a][b][cc] = 0.0f;
    acc.s0 = acc.s1 = acc.s2 = acc.s3 = acc.s4 = make_float2(0.0f, 0.0f);

    double gs0 = 0.0, gs1 = 0.0, gs2 = 0.0, gs3 = 0.0, gs4 = 0.0;  // dense-grid quadrature sums (role 0, inference only)

    // every warp of the CTA walks the same super-tiles (the role barriers need all 4 groups); groups whose
    // 32 points lie beyond n compute on a clamped index with zero weight
    const long long nsuper = (p.n + 127) >> 7;
    int it = 0;
    if (stager) {  // the first super-tile's coordinates (requested before the weight image was built)
      cp_async_wait_all();
      if (tile_bulk(blockIdx.x)) mbar_wait(smem_u32(&cfull[0]), 0u);
    }
    __syncthreads();
    TLK(1);
    // Dense-grid quadrature: R is one number for the whole launch, so E(R) and the gate are too.  The E-net role evaluates
    // them ONCE (through the same tensor-core path, i.e. the same bits every point used to get), leaves them in both mailbox
    // buffers of its group and sits the tile loop out: the two MLP warps of a scheduler have it to themselves (10^8-point
    // quadrature 8.3e9 -> 1.03e10 points/s, same bits).  Letting the idle E-net warps also produce the geometry one tile ahead
    // (filled / consumed barriers, two buffers) is correct and SLOWER, 9.3e9: one producer warp per group with 64-bit index
    // divisions does not keep up with two MLP warps whose inference tile is short.
    // (the spheroidal sweep has one R per super-tile, not per CTA: there the E-net role stays in the tile loop and evaluates
    //  E(R) and the gate per point, as in the fields mode)
    const bool enet_once = !TRAIN && p.grid.on && !p.grid.sph;
    if (enet_once) {
      if (!IS_MLP) {
        const float Rg = (float)p.grid.R;
        float gt;
        const float E = tc_enet_forward<false>(w, c, Rg, Hs + lane * ROWE, Gs + lane * ROWE, sx, gt);
        gbox[2 * 32 + lane] = make_float2(E, gt);
        gbox[3 * 32 + 2 * 32 + lane] = make_float2(E, gt);
        if (blockIdx.x == 0 && grp == 0 && lane == 0) p.grid.partials[8 * (size_t)gridDim.x] = (double)E;  // E(R) of the launch
      }
      named_barrier(1 + grp, (NEV + 1) * 32);
    }
    for (long long st = blockIdx.x; st < nsuper && !(enet_once && !IS_MLP); st += gridDim.x, ++it) {
      const long long pidx = st * 128 + slot;
      const bool valid = pidx < p.n;
      const long long pi = valid ? pidx : (p.n - 1);
      c.tl_it = it;
      TL(0);
      if (it < 38) TLK(2 + it);
      const unsigned char* cbuf = cstage + (it % COORD_STAGES) * COORD_STAGE_BYTES;
      const bool this_bulk = tile_bulk(st);   // (its arrival was awaited by the E-net warps before the last group barrier)
      // The E-net warp (it runs ~2 k cycles ahead of the MLP warps of its group and waits for them mid-tile anyway) forms the
      // geometry of the group's 32 points once and hands it over: the MLP warps - the critical path - start their tile with
      // three 128-bit loads instead of the rsqrt / exp chain (same bits, step -1.5 %: 0.11255 vs 0.11427 ms on one box,
      // profiles/r02_q_ab_geometry_handoff.log).  arrive (E-net) + sync (MLP) on a named barrier per group; two buffers, and
      // the E-net warp cannot be two tiles ahead (mid-tile group barrier).
      // Training launches only: without a reverse sweep the E-net role is not ahead of the MLP roles, and waiting for it
      // cost the 10^8-point grid quadrature 8 % (7.6e9 vs 8.2e9 points/s) - there every role forms its own geometry.
      Geom g;
      float cur_dx1, cur_dx2, mk_f = 0.0f;
      if (!TRAIN) {
        const RawPt raw = p.grid.on ? (p.grid.sph ? tc_sph_point(p.grid, pi) : tc_grid_point(p, pi)) : coord_stage_read(p, cbuf, slot);
        g = geom_from_raw(raw);
        cur_dx1 = raw.dx1; cur_dx2 = raw.dx2;
      } else {
        float4* gp = geo + ((it & 1) * 128 + slot) * 3;
        if (!IS_MLP) {
          const RawPt raw = p.grid.on ? tc_grid_point(p, pi) : coord_stage_read(p, cbuf, slot);
          g = geom_from_raw(raw);
          cur_dx1 = raw.dx1; cur_dx2 = raw.dx2;
          if (TRAIN && p.mask) {  // bulk stage: the 128 mask bytes as they lie; per-lane stage: the aligned word around the byte
            const unsigned mk = this_bulk ? (unsigned)cbuf[4 * COORD_COL_BYTES + slot]
                                          : *(const uint32_t*)(cbuf + 4 * COORD_COL_BYTES + slot * 4) >> (8u * (unsigned)((uintptr_t)(p.mask + pi) & 3u));
            mk_f = (float)(mk & 3u);
          }
          gp[0] = make_float4(g.f1, g.f2, g.ir1, g.ir2);
          gp[1] = make_float4(g.al1, g.al2, g.al11, g.al12);
          gp[2] = make_float4(g.al22, cur_dx1, cur_dx2, mk_f);
          asm volatile("bar.arrive %0, %1;" ::"r"(8 + grp), "r"((NEV + 1) * 32) : "memory");
        } else {
          named_barrier(8 + grp, (NEV + 1) * 32);
          const float4 q0 = gp[0], q1 = gp[1], q2 = gp[2];
          g.f1 = q0.x; g.f2 = q0.y; g.ir1 = q0.z; g.ir2 = q0.w;
          g.al1 = q1.x; g.al2 = q1.y; g.al11 = q1.z; g.al12 = q1.w;
          g.al22 = q2.x; cur_dx1 = q2.y; cur_dx2 = q2.z; mk_f = q2.w;
          g.R = 0.0f;  // only the E-net warp uses R
        }
      }
      if (stager) {  // coordinates of the next super-tile: in flight while this one is computed
        const long long in = pidx + (long long)gridDim.x * 128;
        const long long stn = st + gridDim.x;
        if (stn < nsuper) {
          unsigned char* nbuf = cstage + ((it + 1) % COORD_STAGES) * COORD_STAGE_BYTES;
          if (tile_bulk(stn)) {
            // (training launches only.)  The target buffer was read at the top of the previous super-tile; this thread
            // sits in the E-net role's issuing warp and has since SYNCED on the role barriers of that tile (the other
            // three warps only signal there), i.e. all four E-net warps - the only readers of the stage in training
            // launches - had read their coordinates.
            if (bulk_issuer) coord_stage_issue_bulk(p, nbuf, &cfull[(it + 1) % COORD_STAGES], stn);
          } else {
            coord_stage_issue(p, nbuf, slot, in < p.n ? in : p.n - 1);
          }
        }
        cp_async_commit();
      }
      float2* box = gbox + (it & 1) * (3 * 32);

      // the evaluation at the inversion image swaps the roles of the two nuclei (poc/main.py:255-256)
      const bool sw = (role == 1) && IS_MLP;
      const float a = sw ? g.f2 : g.f1, b = sw ? g.f1 : g.f2;
      const float al1 = sw ? g.al2 : g.al1, al2 = sw ? g.al1 : g.al2;
      const float al11 = sw ? g.al22 : g.al11, al22 = sw ? g.al11 : g.al22;
      const float al12 = g.al12;

      if (IS_MLP) {
        float Nv, Dv;
        tc_mlp_forward<TRAIN>(w, c, cb, a, b, al1, al2, al11, al12, al22, Hs + lane * ROWH, Gs + lane * ROWH, sx, Nv, Dv);
        box[role * 32 + lane] = make_float2(Nv, Dv);
      } else {
        float gt;
        const float E = tc_enet_forward<TRAIN>(w, c, g.R, Hs + lane * ROWE, Gs + lane * ROWE, sx, gt);
        box[2 * 32 + lane] = make_float2(E, gt);
      }
      TL(5);
      if (stager) {  // the NEXT tile's coordinates have landed; the barrier publishes them to the group
        cp_async_wait_all();
        // bulk copies complete on the stage's mbarrier: the E-net warps (the role with slack) wait for it here, off the MLP
        // warps' critical path, and the group barrier hands the data on (use number (it+1)/2 of that stage -> parity)
        const long long stn = st + (long long)gridDim.x;
        if (stn < nsuper && tile_bulk(stn))
          mbar_wait(smem_u32(&cfull[(it + 1) % COORD_STAGES]), (uint32_t)((it + 1) / COORD_STAGES) & 1u);
      }
      named_barrier(1 + grp, enet_once ? NEV * 32 : (NEV + 1) * 32);
      TL(6);

      // ---- combine (every role recomputes the few scalars it needs) ----
      float2 m0 = box[lane];
      if (NEV == 2) { const float2 m1 = box[32 + lane]; m0.x += m1.x; m0.y += m1.y; }
      const float2 me = box[2 * 32 + lane];
      const float E = me.x, gate = me.y;
      const float N = fmaf(sN, m0.x, w.bo), DN = sN * m0.y;
      const float q = g.ir1 + g.ir2;
      const float fs = g.f1 + g.f2;
      const float psi = fmaf(gate, N, fs);
      const float lcao = fmaf(cL, fs, fmaf(cV - 2.0f * cL, fmaf(g.f1, g.ir1, g.f2 * g.ir2),
                                            cV * fmaf(g.f1, g.ir2, g.f2 * g.ir1)));
      const float inner = fmaf(cL, DN, cV * q * N);
      const float res = fmaf(gate, inner, fmaf(cE * E, psi, lcao));

      if (!TRAIN) {
        if (p.grid.sph) {
          // one row per warp of role 0 and super-tile (its 32 points share one R): no state carried across tiles, so the
          // rows of one R are the same bits whatever else the launch sweeps.  Every slot is valid (padded to 128 per R).
          if (role == 0) {
            const double wq = sph_weight(p.grid, pidx);
            const float hl = fmaf(-0.5f, fs, -fmaf(g.f1, g.ir2, g.f2 * g.ir1));
            const float hpsi = fmaf(gate, fmaf(-0.5f, DN, -q * N), hl);
            double v0 = wq * (double)(psi * hpsi), v1 = wq * (double)(psi * psi);
            double v2 = wq * (double)(fs * hl), v3 = wq * (double)(fs * fs);
  #pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
              v0 += __shfl_xor_sync(0xffffffffu, v0, o); v1 += __shfl_xor_sync(0xffffffffu, v1, o);
              v2 += __shfl_xor_sync(0xffffffffu, v2, o); v3 += __shfl_xor_sync(0xffffffffu, v3, o);
            }
            if (lane == 0) {
              double* row = p.grid.partials + 8 * (size_t)(st * 4 + grp);
              row[0] = v0; row[1] = v1; row[2] = v2; row[3] = v3; row[5] = (double)E;
            }
          }
          continue;
        }
        if (p.grid.on) {
          if (valid && role == 0) {
            int ix, iy, iz;
            grid_ijk(p.grid, pi, ix, iy, iz);  // (pi == pidx for a valid point: the same expression as in tc_grid_point above)
            const double wq = p.grid.wx[ix] * p.grid.wy[iy] * p.grid.wz[iz];
            // Hartree form of H psi (poc/main.py:118-120) with the cusp terms cancelled analytically, and its LCAO part
            const float hl = fmaf(-0.5f, fs, -fmaf(g.f1, g.ir2, g.f2 * g.ir1));
            const float hpsi = fmaf(gate, fmaf(-0.5f, DN, -q * N), hl);
            // dV/dR = -(x-R)/r1^3 + (x+R)/r2^3 (poc/main.py:637-642)
            const float vr = fmaf(-cur_dx1, g.ir1 * g.ir1 * g.ir1, cur_dx2 * g.ir2 * g.ir2 * g.ir2);
            gs0 += wq * (double)(psi * hpsi);
            gs1 += wq * (double)(psi * psi);
            gs2 += wq * (double)(fs * hl);
            gs3 += wq * (double)(fs * fs);
            gs4 += wq * (double)(vr * psi * psi);
          }  // (E(R) of the launch was stored behind the partial rows by the E-net role, in front of the loop)
          continue;
        }
        if (valid) {
          if (role == 0) {
            if (p.psi) p.psi[pidx] = psi;
            if (p.lap) p.lap[pidx] = g.al1 + g.al2 + gate * DN;
            if (p.res) p.res[pidx] = res;
            if (p.hpsi)
              p.hpsi[pidx] = fmaf(gate, fmaf(-0.5f, DN, -q * N),
                                  fmaf(-0.5f, fs, -fmaf(g.f1, g.ir2, g.f2 * g.ir1)));
          } else if (!IS_MLP) {
            if (p.E_out) { if (p.E_f64) reinterpret_cast<double*>(p.E_out)[pidx] = (double)E; else p.E_out[pidx] = E; }
          }
        }
        continue;
      }

      // ---- seeds of the reverse sweep (oracle/closed_form.py:loss_and_grad) ----
      float m1f, m2f;
      if (p.mask) {
        const unsigned mk = (unsigned)mk_f;   // the two set bits came with the geometry
        m1f = (mk & 1u) ? 1.0f : 0.0f;
        m2f = (mk & 2u) ? 1.0f : 0.0f;
      } else {
        m1f = (g.ir1 * p.bcut <= 1.0f) ? 1.0f : 0.0f;
        m2f = (g.ir2 * p.bcut <= 1.0f) ? 1.0f : 0.0f;
      }
      const float vw = valid ? 1.0f : 0.0f;
      const float rbar = 2.0f * w_pde * res * vw;
      const float pbar = 2.0f * fmaf(w_bc1, m1f, w_bc2 * m2f) * psi * vw;
      if (IS_MLP) {
        const float lamN = fmaf(rbar, gate * fmaf(cV, q, cE * E), pbar * gate);
        const float lamD = rbar * cL * gate;
        float extra[8];
  #pragma unroll
        for (int i = 0; i < 8; i++) extra[i] = 0.0f;
        if (role == 0) {
          extra[0] = res * res * vw;
          extra[1] = psi * psi * m1f * vw;
          extra[2] = psi * psi * m2f * vw;
          extra[3] = E * vw;
          extra[4] = p.base_grads ? lamN : 0.0f;  // dL/dbo
          extra[5] = m1f * vw;
          extra[6] = m2f * vw;
        }
        if (p.base_grads) {
          tc_mlp_backward(w, c, cb, a, b, al1, al2, al11, al12, al22, sN * lamN, sN * lamD, Hs, Gs, lane, extra, acc);
        } else if (role == 0) {
          tc_mlp_extras_only(Hs, lane, extra, acc);
        }
      } else {
        if (valid && p.E_out) { if (p.E_f64) reinterpret_cast<double*>(p.E_out)[pidx] = (double)E; else p.E_out[pidx] = E; }
        const float gbar = fmaf(rbar, fmaf(cE * E, N, inner), pbar * N);
        const float Ebar = rbar * cE * psi;
        tc_enet_backward(w, c, g.R, Ebar, gbar, p.gate_grads != 0, Hs, Gs, lane, acc);
      }
      TL(15);
    }

    TLK(40);
    if (TRAIN && blockIdx.x == 0 && tid == 0) {  // (tid 0 is an MLP thread of role 0; both branches run this lambda)
      unsigned long long ns1;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns1));
      double* tm = reinterpret_cast<double*>(mbox);  // the mailbox is free after the last super-tile
      tm[0] = (double)((uint32_t)clock() - *clk0_slot);   // 32-bit cycle counter: differences are exact modulo 2^32
      tm[1] = (double)(ns1 - *ns0_slot);
    }
    // the reduction kernel behind this launch may be set up now (it waits for this grid to complete before it reads)
    pdl_launch_dependents();
    // ---- teardown of tensor memory: all tcgen05 traffic of the CTA is complete (every MMA was waited for) ----
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
      tc_fence_after();
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(c.tbase) : "memory");
    }
    if (!TRAIN) {
      if (p.grid.on && !p.grid.sph) {  // one row of quadrature sums per CTA, fixed order
        double* red = reinterpret_cast<double*>(stash);
        if (role == 0) {
  #pragma unroll
          for (int o = 16; o > 0; o >>= 1) {
            gs0 += __shfl_xor_sync(0xffffffffu, gs0, o); gs1 += __shfl_xor_sync(0xffffffffu, gs1, o);
            gs2 += __shfl_xor_sync(0xffffffffu, gs2, o); gs3 += __shfl_xor_sync(0xffffffffu, gs3, o);
            gs4 += __shfl_xor_sync(0xffffffffu, gs4, o);
          }
          if (lane == 0) { red[grp * 8 + 0] = gs0; red[grp * 8 + 1] = gs1; red[grp * 8 + 2] = gs2; red[grp * 8 + 3] = gs3; red[grp * 8 + 4] = gs4; }
        }
        __syncthreads();
        if (tid < 5) p.grid.partials[8 * (size_t)blockIdx.x + tid] = (red[tid] + red[8 + tid]) + (red[16 + tid] + red[24 + tid]);
      }
      return;
    }

    // ---- fold: every warp writes its accumulators into its own row of floats (the stash is free now), then all
    //      threads add the rows entry by entry in a fixed order, in double -> one deterministic row per CTA ----
    {
      // (no zero fill: every MLP warp writes all base-MLP entries, role 0 also bo and the loss sums, every E-net warp
      // all E-net and gate entries; the final sum below only reads the rows of the warps that own an entry)
      float* myrow = stash + warp * NPART;
      const int gq = lane >> 2, tq = lane & 3;
      if (IS_MLP) {
  #pragma unroll
        for (int nt = 0; nt < 2; nt++) {
          const int j0 = gq, j1 = gq + 8, k0 = nt * 8 + 2 * tq, k1 = k0 + 1;
          myrow[O_W2 + j0 * NH + k0] = acc.c[0][nt][0] + acc.c[1][nt][0];
          myrow[O_W2 + j0 * NH + k1] = acc.c[0][nt][1] + acc.c[1][nt][1];
          myrow[O_W2 + j1 * NH + k0] = acc.c[0][nt][2] + acc.c[1][nt][2];
          myrow[O_W2 + j1 * NH + k1] = acc.c[0][nt][3] + acc.c[1][nt][3];
        }
        // window index i (0..31) of each vector sum -> entry of the row
        auto e0 = [](int i) { return i < 16 ? O_B2 + i : O_WO + i - 16; };
        auto e1 = [](int i) { return i < 16 ? O_W1 + 2 * i : O_W1 + 2 * (i - 16) + 1; };
        auto e2 = [role](int i) {
          if (i < 16) return (int)O_B1 + i;
          if (role != 0) return -1;
          const int e = i - 16;
          return e == 0 ? (int)S_RES2 : e == 1 ? (int)S_PSI1 : e == 2 ? (int)S_PSI2 : e == 3 ? (int)S_E
               : e == 4 ? (int)O_BO : e == 5 ? (int)S_CNT1 : e == 6 ? (int)S_CNT2 : -1;
        };
        fold_pair(myrow, acc.s0, lane, e0);
        fold_pair(myrow, acc.s1, lane, e1);
        fold_pair(myrow, acc.s2, lane, e2);
      } else {
  #pragma unroll
        for (int mt = 0; mt < 2; mt++)
  #pragma unroll
          for (int nt = 0; nt < 4; nt++) {
            const int j0 = mt * 16 + gq, j1 = j0 + 8, k0 = nt * 8 + 2 * tq, k1 = k0 + 1;
            myrow[O_WE2 + j0 * NE + k0] = acc.c[mt][nt][0];
            myrow[O_WE2 + j0 * NE + k1] = acc.c[mt][nt][1];
            myrow[O_WE2 + j1 * NE + k0] = acc.c[mt][nt][2];
            myrow[O_WE2 + j1 * NE + k1] = acc.c[mt][nt][3];
          }
        fold_pair(myrow, acc.s0, lane, [](int i) { return (int)O_WE + i; });
        fold_pair(myrow, acc.s1, lane, [](int i) { return (int)O_BE2 + i; });
        fold_pair(myrow, acc.s2, lane, [](int i) { return (int)O_WE1 + i; });
        fold_pair(myrow, acc.s3, lane, [](int i) { return (int)O_BE1 + i; });
        fold_pair(myrow, acc.s4, lane, [](int i) {
          return i < 10 ? (int)O_WGL + i : i < 20 ? (int)O_BGL + i - 10 : i < 30 ? (int)O_WG + i - 20 : i == 30 ? (int)O_BG : (int)O_BE;
        });
      }
    }
    __syncthreads();
    constexpr int nwarps = (NEV + 1) * G;
    double* row = p.partials + (size_t)blockIdx.x * NPART;
    for (int i = tid; i < NPART; i += blockDim.x) {
      // owners of entry i: base-MLP weights <- all MLP warps; bo and the loss sums <- role 0; E-net and gate <- E-net warps
      int w0, w1;
      if (i < O_BO) { w0 = 0; w1 = NEV * G; }
      else if (i == O_BO || (i >= S_RES2 && i <= S_CNT2)) { w0 = 0; w1 = G; }
      else if (i < NTHETA) { w0 = NEV * G; w1 = nwarps; }
      else { w0 = 0; w1 = 0; }  // padding
      double sum = 0.0;
      for (int wv = w0; wv < w1; wv++) sum += (double)stash[wv * NPART + i];
      if (i >= NPART - 2 && blockIdx.x == 0) sum = reinterpret_cast<const double*>(mbox)[i - (NPART - 2)];  // CTA 0's own timing
      row[i] = sum;
    }
    TLK(41);
  };
  constexpr bool REBALANCE = TRAIN && NEV == 2;  // 3 warpgroups at 168 registers: 128 * REG_ENET + 256 * REG_MLP = 384 * 168
  if (is_mlp) {
    if constexpr (REBALANCE) asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(TC_REG_MLP));
    run_role(std::true_type{});
  } else {
    if constexpr (REBALANCE) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(TC_REG_ENET));
    run_role(std::false_type{});
  }
}

// =================================================================================================
// host-side launcher
// =================================================================================================
template <int NEV, bool TRAIN, bool INLINE>
static cudaError_t launch_step_tc_t(const StepParams& p, int grid, cudaStream_t st) {
  auto kern = pinn_step_tc_kernel<NEV, TRAIN, INLINE>;
  constexpr size_t smem = tc_smem_bytes<NEV>();
  static bool configured[16] = {false};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 16 && !configured[dev]) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    configured[dev] = true;
  }
  if constexpr (INLINE) {
    TcParamsInline q;
    q.p = p;
    memcpy(q.theta, p.theta_inline, NTHETA * sizeof(float));
    q.theta[NTHETA] = q.theta[NTHETA + 1] = q.theta[NTHETA + 2] = 0.0f;
    q.w[0] = q.w[1] = q.w[2] = q.w[3] = 0.0;
    if (p.weights_inline) memcpy(q.w, p.weights_inline, 3 * sizeof(double));
    q.p.w_by_value = p.weights_inline != nullptr;
    return launch_pdl(kern, dim3(grid), dim3((NEV + 1) * 128), smem, st, q);
  } else {
    TcParamsPlain q;
    q.p = p;
    q.w[0] = q.w[1] = q.w[2] = q.w[3] = 0.0;
    if (p.weights_inline) memcpy(q.w, p.weights_inline, 3 * sizeof(double));
    q.p.w_by_value = p.weights_inline != nullptr;
    return launch_pdl(kern, dim3(grid), dim3((NEV + 1) * 128), smem, st, q);
  }
}

// adds the per-CTA quadrature rows in a fixed order; out[5] = E(R) stored behind the rows
__global__ void grid_finish_kernel(const double* __restrict__ partials, int nrows, double* __restrict__ out) {
  const int t = threadIdx.x;
  if (t < 5) {
    double s = 0.0;
    for (int r = 0; r < nrows; r++) s += partials[8 * (size_t)r + t];
    out[t] = s;
  } else if (t == 5) {
    out[5] = partials[8 * (size_t)nrows];
  } else if (t < 8) {
    out[t] = 0.0;
  }
}
cudaError_t launch_grid_finish(const double* partials, int nrows, double* out, cudaStream_t st) {
  grid_finish_kernel<<<1, 32, 0, st>>>(partials, nrows, out);
  return cudaGetLastError();
}

// one thread per (R, slot): the rows of one R added in row order (tile-major, then group), E(R) from its first row
__global__ void sph_finish_kernel(const double* __restrict__ partials, int nR, int rows_per_R, const double* __restrict__ Rs,
                                  double* __restrict__ out) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= 8ll * nR) return;
  const int k = (int)(t >> 3), slot = (int)(t & 7);
  const double* rows = partials + 8 * (size_t)k * rows_per_R;
  double v = 0.0;
  if (slot < 4) {
    for (int r = 0; r < rows_per_R; r++) v += rows[8 * (size_t)r + slot];
  } else if (slot == 5) {
    v = rows[5];
  }
  if (!(Rs[k] > 0.0)) v = __longlong_as_double(0x7ff8000000000000ll);  // R <= 0 is no molecule: a NaN row, never numbers
  out[t] = v;
}
cudaError_t launch_sph_finish(const double* partials, int nR, int rows_per_R, const double* Rs, double* out, cudaStream_t st) {
  const long long n = 8ll * nR;
  sph_finish_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(partials, nR, rows_per_R, Rs, out);
  return cudaGetLastError();
}

cudaError_t launch_step_tc(int nev, bool train, const StepParams& p, int grid, cudaStream_t st) {
  if (train && p.theta_inline)
    return nev == 2 ? launch_step_tc_t<2, true, true>(p, grid, st) : launch_step_tc_t<1, true, true>(p, grid, st);
  if (nev == 2) return train ? launch_step_tc_t<2, true, false>(p, grid, st) : launch_step_tc_t<2, false, false>(p, grid, st);
  return train ? launch_step_tc_t<1, true, false>(p, grid, st) : launch_step_tc_t<1, false, false>(p, grid, st);
}

}  // namespace pinn
