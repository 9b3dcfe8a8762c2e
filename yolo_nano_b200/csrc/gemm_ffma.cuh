// fp32 CUDA-core (FFMA) contraction kernels: pointwise 1x1 conv and dense 3x3 conv as an
// implicit GEMM over NHWC pixels.  This is the cross-check path (YNB_GEMM_FP32_FFMA):
// exact fp32 accumulation, used to validate the tcgen05 kernels on the device and as the
// fp32 reference mode; the tensor-core kernels in gemm_tc.cuh are the product path.
//
//   D[m, n] = act(bias[n] + sum_k A[m, k] * W[n, k])
//   A: NHWC pixels x channels (K-major), W: [N][K] K-major (PyTorch [cout][cin] order).
#pragma once
#include "common.cuh"

namespace ynb {

struct GemmParams {
  // A operand
  const float* a;
  int a_ld, a_off;
  // optional second operand added on the fly (3x3 path): A = a + resample(a2)
  //   a2_mode 0: none, 1: nearest up x2 (a2 is H/2 x W/2), 2: nearest down x0.5 (a2 is 2H x 2W)
  //   (models/yolo_nano.py:291-296, F.interpolate default 'nearest')
  const float* a2;
  int a2_ld, a2_mode;
  int H, W;          // spatial size of the output map (3x3 path)
  int C;             // channels per tap (3x3 path), multiple of 16
  // weights / bias
  const float* w;    // [N][Ktot]
  const float* bias; // [N]
  // output
  float* out;
  int out_ld, out_off, out_step;
  int64_t M;
  int N, Ktot;       // Ktot multiple of 4
  int act;
};

template <int BN, bool K3X3>
__global__ void __launch_bounds__(256)
gemm_ffma_kernel(GemmParams p) {
  constexpr int BM = 128, BK = 16, TN = BN / 16;
  __shared__ __align__(16) float As[BK][BM + 4];
  __shared__ __align__(16) float Bs[BK][BN + 4];

  const int tid = threadIdx.x;
  const int64_t m0 = (int64_t)blockIdx.x * BM;
  const int n0 = blockIdx.y * BN;
  const int ty = tid >> 4, tx = tid & 15;

  // A loader: 2 float4 per thread; rows fixed across the K loop
  int a_row[2], a_kq[2];
  int64_t a_pix[2];              // pixel index (pointwise) / base pixel of the image (3x3)
  int a_y[2], a_x[2];
  bool a_ok[2];
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    int idx = tid + i * 256;
    a_row[i] = idx >> 2;
    a_kq[i] = idx & 3;
    int64_t m = m0 + a_row[i];
    a_ok[i] = m < p.M;
    if (K3X3) {
      int64_t hw = (int64_t)p.H * p.W;
      int64_t b = a_ok[i] ? m / hw : 0;
      int r = a_ok[i] ? (int)(m - b * hw) : 0;
      a_y[i] = r / p.W;
      a_x[i] = r - a_y[i] * p.W;
      a_pix[i] = b;
    } else {
      a_pix[i] = m;
      a_y[i] = a_x[i] = 0;
    }
  }
  // B loader
  constexpr int B_F4 = BN * 4;                 // float4 per tile
  constexpr int B_PER = (B_F4 + 255) / 256;

  float acc[8][TN];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.0f;

  float4 ra[2], rb[B_PER];

  auto load_tiles = [&](int k0) {
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      int k = k0 + 4 * a_kq[i];
      if (a_ok[i] && k < p.Ktot) {
        if (K3X3) {
          int tap = k / p.C;
          int c = k - tap * p.C;
          int dy = tap / 3, dx = tap - dy * 3;
          int y = a_y[i] + dy - 1, x = a_x[i] + dx - 1;
          if (y >= 0 && y < p.H && x >= 0 && x < p.W) {
            size_t pix = ((size_t)a_pix[i] * p.H + y) * p.W + x;
            v = __ldg(reinterpret_cast<const float4*>(p.a + pix * p.a_ld + p.a_off + c));
            if (p.a2_mode == 1) {
              int H2 = p.H >> 1, W2 = p.W >> 1;
              size_t q = ((size_t)a_pix[i] * H2 + (y >> 1)) * W2 + (x >> 1);
              float4 u = __ldg(reinterpret_cast<const float4*>(p.a2 + q * p.a2_ld + c));
              v.x += u.x; v.y += u.y; v.z += u.z; v.w += u.w;
            } else if (p.a2_mode == 2) {
              int H2 = p.H << 1, W2 = p.W << 1;
              size_t q = ((size_t)a_pix[i] * H2 + (y << 1)) * W2 + (x << 1);
              float4 u = __ldg(reinterpret_cast<const float4*>(p.a2 + q * p.a2_ld + c));
              v.x += u.x; v.y += u.y; v.z += u.z; v.w += u.w;
            }
          }
        } else {
          v = __ldg(reinterpret_cast<const float4*>(p.a + (size_t)a_pix[i] * p.a_ld + p.a_off + k));
        }
      }
      ra[i] = v;
    }
#pragma unroll
    for (int i = 0; i < B_PER; ++i) {
      int idx = tid + i * 256;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (idx < B_F4) {
        int n = n0 + (idx >> 2);
        int k = k0 + 4 * (idx & 3);
        if (n < p.N && k < p.Ktot) v = __ldg(reinterpret_cast<const float4*>(p.w + (size_t)n * p.Ktot + k));
      }
      rb[i] = v;
    }
  };
  auto store_tiles = [&]() {
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      int kq = 4 * a_kq[i];
      As[kq + 0][a_row[i]] = ra[i].x;
      As[kq + 1][a_row[i]] = ra[i].y;
      As[kq + 2][a_row[i]] = ra[i].z;
      As[kq + 3][a_row[i]] = ra[i].w;
    }
#pragma unroll
    for (int i = 0; i < B_PER; ++i) {
      int idx = tid + i * 256;
      if (idx < B_F4) {
        int n = idx >> 2, kq = 4 * (idx & 3);
        Bs[kq + 0][n] = rb[i].x;
        Bs[kq + 1][n] = rb[i].y;
        Bs[kq + 2][n] = rb[i].z;
        Bs[kq + 3][n] = rb[i].w;
      }
    }
  };

  load_tiles(0);
  for (int k0 = 0; k0 < p.Ktot; k0 += BK) {
    __syncthreads();
    store_tiles();
    __syncthreads();
    if (k0 + BK < p.Ktot) load_tiles(k0 + BK);
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      float4 a0 = *reinterpret_cast<const float4*>(&As[k][ty * 8]);
      float4 a1 = *reinterpret_cast<const float4*>(&As[k][ty * 8 + 4]);
      float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      float bv[TN];
#pragma unroll
      for (int j = 0; j < TN; ++j) bv[j] = Bs[k][tx + 16 * j];
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
  }

#pragma unroll
  for (int j = 0; j < TN; ++j) {
    int n = n0 + tx + 16 * j;
    if (n >= p.N) continue;
    float bj = __ldg(p.bias + n);
    int col = p.out_off + n * p.out_step;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      int64_t m = m0 + ty * 8 + i;
      if (m < p.M) p.out[m * p.out_ld + col] = apply_act(acc[i][j] + bj, p.act);
    }
  }
}

inline cudaError_t launch_gemm_ffma(const GemmParams& p, bool k3x3, cudaStream_t st) {
  if (p.M <= 0) return cudaSuccess;
  unsigned mt = (unsigned)((p.M + 127) / 128);
  // N tile: 58 -> 64, 96 -> 96, 116 -> 2 x 64, 232 / 255 -> 2 x 128
  int bn = p.N <= 64 ? 64 : (p.N <= 96 ? 96 : (p.N <= 128 ? 64 : 128));
  dim3 grid(mt, (p.N + bn - 1) / bn);
#define YNB_GEMM_LAUNCH(BN_)                                              \
  do {                                                                    \
    if (k3x3) gemm_ffma_kernel<BN_, true><<<grid, 256, 0, st>>>(p);       \
    else gemm_ffma_kernel<BN_, false><<<grid, 256, 0, st>>>(p);           \
  } while (0)
  if (bn == 64) YNB_GEMM_LAUNCH(64);
  else if (bn == 96) YNB_GEMM_LAUNCH(96);
  else YNB_GEMM_LAUNCH(128);
#undef YNB_GEMM_LAUNCH
  YNB_COUNT_LAUNCH();
  return cudaGetLastError();
}

}  // namespace ynb
