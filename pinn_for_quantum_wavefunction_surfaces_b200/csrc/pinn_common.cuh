// Shared constants and small device helpers of the PINN hot-path kernels (sm_100a).
#pragma once
#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>

namespace pinn {

constexpr int NH = 16;   // base-MLP hidden width   (poc/main.py:227; train.py:85)
constexpr int NE = 32;   // E-net hidden width      (poc/main.py:228; train.py:86)
constexpr int NL = 10;   // gate hidden width       (poc/main.py:229; train.py:87)
constexpr int NTHETA = 1521;
constexpr int NPART = 1536;  // one row of partial sums: 1521 gradients + 8 loss sums, padded

// offsets inside theta (state_dict order, SURVEY.md Appendix B)
enum : int {
  O_W1 = 0, O_B1 = 32, O_W2 = 48, O_B2 = 304, O_WO = 320, O_BO = 336,
  O_WE1 = 337, O_BE1 = 369, O_WE2 = 401, O_BE2 = 1425, O_WE = 1457, O_BE = 1489,
  O_WGL = 1490, O_BGL = 1500, O_WG = 1510, O_BG = 1520,
  // loss sums ride behind the gradients in a partial row
  S_RES2 = 1521, S_PSI1 = 1522, S_PSI2 = 1523, S_E = 1524, S_CNT1 = 1525, S_CNT2 = 1526
};

// Weights as the step kernel wants them: every CTA builds this image in its shared memory from theta
// (build_weight_image, pinn_device.cuh).
struct alignas(128) Wts {
  float w0[NH], w1[NH], b1[NH];          // W1[:,0], W1[:,1], b1
  float ww00[NH], ww01[NH], ww11[NH];    // w0^2, w0*w1, w1^2  (second-order channel)
  float b2[NH], wo[NH];
  float WE1[NE], bE1[NE];
  float bE2[NE], wE[NE];
  float WgL[12], bgL[12], wg[12];        // 10 used
  float bo, bE, bg, pad0;
  float w0s[NH], w1s[NH], b1s[NH], b2s[NH];  // w0, w1, b1, b2 times -log2(e): pre-activations arrive as the MUFU.EX2 argument
  float WE1s[NE], bE1s[NE], bE2s[NE];    // the same for the E-net ...
  float WgLs[12], bgLs[12];              // ... and the gate (10 used); 480 floats so far: the images below stay 128-byte aligned
  // ---- tcgen05 B operands (pinn_step_tc.cu): [hi | lo] TF32 split, K-major canonical no-swizzle layout
  //      (8-row x 16-byte core matrices; see umma_off()) ----
  float BS[2][NH * NH];                  // n = j        : W2[j][k]                      (A = s)
  float BSP[2][2 * NH * NH];             // n = c*16 + j : W2[j][k] * {w0,w1}[k]         (A = s')
  float BSPP[2][3 * NH * NH];            // n = c*16 + j : W2[j][k] * {w0^2,w0w1,w1^2}[k] (A = s'')
  float BWT[2][NH * NH];                 // n = k        : W2[j][k], K index = j          (reverse sweep)
  float BE[2][NE * NE];                  // n = j        : WE2[j][k]
  float BET[2][NE * NE];                 // n = k        : WE2[j][k], K index = j
};
// offset (floats) of element (n,k) of an N x K operand in the canonical K-major no-swizzle layout:
// 16-byte K chunks strided by LBO = 128*(N/8) bytes, 8-row groups strided by SBO = 128 bytes
__host__ __device__ constexpr int umma_off(int n, int k, int N) {
  return (k / 4) * (32 * (N / 8)) + (n / 8) * 32 + (n % 8) * 4 + (k % 4);
}
static_assert(sizeof(Wts) == 32640, "Wts: 480 layer floats + the six hi/lo operand images");
static_assert(offsetof(Wts, BS) % 128 == 0 && sizeof(Wts) % 128 == 0,
              "operand images and the shared-memory buffers behind the image must stay aligned");

// entry i of the canonical theta -> index inside ITS tensor when that tensor is stored in train.py's (in,out) layout
// (x @ A + b, train.py:4-5) instead of nn.Linear's (out,in); only W1 (16,2), W2 (16,16) and WE2 (32,32) differ
__host__ __device__ constexpr int in_out_index(int tensor, int j) {
  return tensor == 0 ? (j % 2) * NH + j / 2 : tensor == 2 ? (j % NH) * NH + j / NH : tensor == 8 ? (j % NE) * NE + j / NE : j;
}
// tensor index k (state_dict order) and start offset of entry i of theta - compare/select chains on immediates (an
// offset table indexed at run time would live on the thread's stack)
__host__ __device__ inline void theta_locate(int i, int& k, int& off) {
  k = 0; off = O_W1;
#define PINN_T(K, O) if (i >= (O)) { k = (K); off = (O); }
  PINN_T(1, O_B1) PINN_T(2, O_W2) PINN_T(3, O_B2) PINN_T(4, O_WO) PINN_T(5, O_BO) PINN_T(6, O_WE1) PINN_T(7, O_BE1)
  PINN_T(8, O_WE2) PINN_T(9, O_BE2) PINN_T(10, O_WE) PINN_T(11, O_BE) PINN_T(12, O_WGL) PINN_T(13, O_BGL) PINN_T(14, O_WG)
  PINN_T(15, O_BG)
#undef PINN_T
}

struct VariantCoef {  // res = cL*lap(psi) + cV*(1/r1+1/r2)*psi + cE*E*psi ; N = sN * sum(evals) + bo
  float sN, cL, cV, cE;
};

}  // namespace pinn
