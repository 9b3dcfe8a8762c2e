// HBM-bound kernels of the path: stem conv + max-pool, depthwise 3x3, pass-through
// interleave (channel shuffle as a store permutation) and layout conversion for taps.
#pragma once
#include <algorithm>
#include "common.cuh"
#include "ptx_sm100.cuh"

namespace ynb {

// =====================================================================================
// Stem: Conv2d(3,24,3,s2,p1, no bias)+BN(folded)+ReLU -> MaxPool2d(3,s2,p1), one kernel.
// (backbone/shufflenetv2.py:109-116,158-159)
//   x   NCHW [B,3,S,S]      out NHWC [B,S/4,S/4,24]
//   w   [27][24], index (ci*9 + ky*3 + kx)*24 + co     b [24]
// A CTA owns an 8x8 tile of pooled outputs: 17x17 conv outputs, 35x35x3 input pixels.
// The 24x208x208 conv map (the largest tensor of the network) never reaches HBM.
// MaxPool pads with -inf; conv outputs are post-ReLU (>= 0) and every pooling window holds
// at least one valid element, so padding with 0 gives the same maximum.
// =====================================================================================
constexpr int kStemTile = 8;
constexpr int kStemConv = 2 * kStemTile + 1;   // 17
constexpr int kStemIn = 2 * kStemConv + 1;     // 35
constexpr int kStemInPitch = 40;               // TMA box rows: 40 floats; the box starts ONE column left of the
                                               // patch so that its first element is 16-byte aligned in global memory
constexpr int kStemC = 24;
constexpr int kStemCP = 24;                    // s_conv pitch: 16-byte aligned rows, 45.5 KB static smem in total
constexpr int kStemPairs = (kStemConv + 1) / 2;                  // 9 column pairs per conv row
constexpr int kStemTasks2 = kStemConv * kStemPairs;              // (row, column pair) = 153, all 24 channels each
constexpr int kStemThreads = 160;

// Folded stem weights travel as a kernel parameter (constant bank) and are staged in shared
// memory by every CTA.
struct StemWeights {
  float w[27][kStemC];   // [(ci*3+ky)*3+kx][co]
  float b[kStemC];
};

// Input patch: ONE TMA box load per CTA — [40 x 35 x 3] floats of the NCHW image at (ix0 - 1, iy0),
// out-of-image elements zero-filled by the copy engine (= the conv's zero padding) — instead of
// twelve bounds-checked scalar loads per thread.  tmX == nullptr-equivalent (use_tma = 0, input
// not 16-byte aligned) falls back to those loads.
//
// The conv is bound by the FMA pipe / issue slots (648 FMAs per conv output), so it is written
// with the packed FFMA2 (two fp32 FMAs per instruction, each rounded exactly like fmaf): a thread
// owns two horizontally adjacent conv positions and 12 of the 24 output channels = 12 float2
// accumulators; per tap it reads two input pixels and three 16-byte weight vectors (broadcast)
// and issues 12 FFMA2.  (Measured on B200, tools/fma_probe.cu: FFMA with a constant-bank /
// uniform-register operand runs at half rate, which is what the previous version did.)
template <typename OutT>
__global__ void __launch_bounds__(kStemThreads)
stem_pool_kernel(const float* __restrict__ x, OutT* __restrict__ out, const __grid_constant__ StemWeights wt,
                 const __grid_constant__ CUtensorMap tmX, int use_tma, int S) {
  __shared__ __align__(128) float s_in[3][kStemIn][kStemInPitch];
  __shared__ __align__(16) float s_conv[kStemConv * kStemConv][kStemCP];
  __shared__ __align__(8) uint64_t s_bar;

  const int Hc = S / 2, Hp = S / 4;
  const int b = blockIdx.z;
  const int py0 = blockIdx.y * kStemTile, px0 = blockIdx.x * kStemTile;
  const int cy0 = 2 * py0 - 1, cx0 = 2 * px0 - 1;   // first conv row / col of the tile
  const int iy0 = 2 * cy0 - 1, ix0 = 2 * cx0 - 1;   // first input row / col
  const int tid = threadIdx.x;
  pdl_trigger();
  if (use_tma && tid == 0) {
    ptx::mbar_init(&s_bar, 1);
    ptx::fence_barrier_init();
  }
  pdl_wait();          // the previous forward may still be reading / writing these buffers

  if (use_tma) {
    if (tid == 0) {
      ptx::mbar_arrive_expect_tx(&s_bar, 3 * kStemIn * kStemInPitch * 4);
      ptx::tma_load_4d(&s_in[0][0][0], &tmX, &s_bar, ix0 - 1, iy0, 0, b);   // 16*bx - 4: multiple of 4 floats
    }
    __syncthreads();                                   // barrier init visible + weights staged
    ptx::mbar_wait(&s_bar, 0, nullptr, 0);
  } else {
    const float* xb = x + (size_t)b * 3 * S * S;
    for (int i = tid; i < 3 * kStemIn * kStemIn; i += kStemThreads) {
      const int c = i / (kStemIn * kStemIn);
      const int rem = i - c * (kStemIn * kStemIn);
      const int r = rem / kStemIn, q = rem - r * kStemIn;
      const int iy = iy0 + r, ix = ix0 + q;
      float v = 0.0f;
      if (iy >= 0 && iy < S && ix >= 0 && ix < S) v = __ldg(xb + ((size_t)c * S + iy) * S + ix);
      s_in[c][r][q + 1] = v;
    }
    __syncthreads();
  }

  // conv + bias + ReLU.  Round 2: the kernel was bound by the shared-memory pipe (ncu l1tex 96 %): a broadcast
  // LDS.128 of weights still costs four wavefronts per warp and there were 81 of them per thread.  The weights now
  // come straight from the constant bank (the kernel parameter) as FFMA operands — half the FMA issue rate
  // (tools/fma_probe.cu: 65 vs 126 FMA/clk/SM) but no shared-memory traffic at all; a thread owns two horizontally
  // adjacent conv positions and ALL 24 output channels (48 accumulators), every constant feeds both positions.
  if (tid < kStemTasks2) {
    const int r = tid / kStemPairs, q0 = (tid - r * kStemPairs) * 2;
    const bool has2 = q0 + 1 < kStemConv;
    float acc0[kStemC], acc1[kStemC];
#pragma unroll
    for (int j = 0; j < kStemC; ++j) acc0[j] = acc1[j] = wt.b[j];
#pragma unroll
    for (int ci = 0; ci < 3; ++ci)
#pragma unroll
      for (int ky = 0; ky < 3; ++ky) {
        const float* row = &s_in[ci][2 * r + ky][1];
        float in[5];
#pragma unroll
        for (int j = 0; j < 5; ++j) in[j] = row[min(2 * q0 + j, kStemIn - 1)];
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
#pragma unroll
          for (int j = 0; j < kStemC; ++j) {
            const float w = wt.w[(ci * 3 + ky) * 3 + kx][j];
            acc0[j] = fmaf(in[kx], w, acc0[j]);
            acc1[j] = fmaf(in[kx + 2], w, acc1[j]);
          }
        }
      }
    const int cy = cy0 + r;
    const bool row_in = cy >= 0 && cy < Hc;
    const bool in0 = row_in && cx0 + q0 >= 0 && cx0 + q0 < Hc;
    const bool in1 = row_in && cx0 + q0 + 1 >= 0 && cx0 + q0 + 1 < Hc;
    float4* d0 = reinterpret_cast<float4*>(&s_conv[r * kStemConv + q0][0]);
#pragma unroll
    for (int j = 0; j < kStemC / 4; ++j)
      d0[j] = in0 ? make_float4(fmaxf(acc0[4 * j], 0.f), fmaxf(acc0[4 * j + 1], 0.f), fmaxf(acc0[4 * j + 2], 0.f),
                                fmaxf(acc0[4 * j + 3], 0.f))
                  : make_float4(0.f, 0.f, 0.f, 0.f);
    if (has2) {
      float4* d1 = reinterpret_cast<float4*>(&s_conv[r * kStemConv + q0 + 1][0]);
#pragma unroll
      for (int j = 0; j < kStemC / 4; ++j)
        d1[j] = in1 ? make_float4(fmaxf(acc1[4 * j], 0.f), fmaxf(acc1[4 * j + 1], 0.f), fmaxf(acc1[4 * j + 2], 0.f),
                                  fmaxf(acc1[4 * j + 3], 0.f))
                    : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
  __syncthreads();

  // 3x3 / stride 2 max-pool: a thread takes 4 channels of one pooled pixel (16-byte accesses)
  for (int i = tid; i < kStemTile * kStemTile * (kStemC / 4); i += kStemThreads) {
    const int p = i / (kStemC / 4), c4 = (i - p * (kStemC / 4)) * 4;
    const int r = p / kStemTile, q = p - r * kStemTile;
    const int py = py0 + r, px = px0 + q;
    if (py >= Hp || px >= Hp) continue;
    float4 m = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int dy = 0; dy < 3; ++dy)
#pragma unroll
      for (int dx = 0; dx < 3; ++dx) {
        const float4 v = *reinterpret_cast<const float4*>(&s_conv[(2 * r + dy) * kStemConv + 2 * q + dx][c4]);
        m.x = fmaxf(m.x, v.x); m.y = fmaxf(m.y, v.y); m.z = fmaxf(m.z, v.z); m.w = fmaxf(m.w, v.w);
      }
    store4(out + (((size_t)b * Hp + py) * Hp + px) * kStemC + c4, m);
  }
}

// tmX: rank-4 map over the NCHW input (make_tmap_stem_input); pass use_tma = 0 (any map) when the
// input pointer is not 16-byte aligned.
inline cudaError_t launch_stem_pool(const float* x, void* out, bool out_bf16, const StemWeights& wt,
                                    const CUtensorMap& tmX, int use_tma, int batch, int S, cudaStream_t st) {
  int Hp = S / 4;
  dim3 grid((Hp + kStemTile - 1) / kStemTile, (Hp + kStemTile - 1) / kStemTile, batch);
  cudaError_t r = out_bf16
      ? launch_pdl(stem_pool_kernel<bf16>, grid, dim3(kStemThreads), 0, st, x, static_cast<bf16*>(out), wt, tmX, use_tma, S)
      : launch_pdl(stem_pool_kernel<float>, grid, dim3(kStemThreads), 0, st, x, static_cast<float*>(out), wt, tmX, use_tma, S);
  YNB_COUNT_LAUNCH();
  return r;
}

// =====================================================================================
// Test-time augmentation input (SURVEY §8f row 2; utils/misc.py:104-121): bilinear resize of the
// NCHW input to s x s with align_corners=False (torch.nn.functional.interpolate) and, optionally, the
// horizontally flipped copy (torch.flip(x, [-1])) — written as out[2b] = resized, out[2b+1] = flipped.
//   src = (dst + 0.5) * (in / out) - 0.5, clamped at 0; neighbours clamped at in - 1
//   out = (1-ly) * ((1-lx) v00 + lx v01) + ly * ((1-lx) v10 + lx v11)
// =====================================================================================
__global__ void __launch_bounds__(256)
resize_bilinear_kernel(const float* __restrict__ in, float* __restrict__ out, int planes, int Hi, int Wi, int So,
                       int with_flip) {
  const int64_t total = (int64_t)planes * So * So;
  const float sy = (float)Hi / (float)So, sx = (float)Wi / (float)So;
  pdl_trigger();
  pdl_wait();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int ox = (int)(i % So);
    const int oy = (int)((i / So) % So);
    const int64_t pl = i / ((int64_t)So * So);                 // b * C + c
    const float fy = fmaxf(sy * ((float)oy + 0.5f) - 0.5f, 0.0f), fx = fmaxf(sx * ((float)ox + 0.5f) - 0.5f, 0.0f);
    const int y0 = min((int)fy, Hi - 1), x0 = min((int)fx, Wi - 1);
    const int y1 = min(y0 + 1, Hi - 1), x1 = min(x0 + 1, Wi - 1);
    const float ly = fy - (float)y0, lx = fx - (float)x0;
    const float* src = in + pl * Hi * Wi;
    const float v00 = __ldg(src + y0 * Wi + x0), v01 = __ldg(src + y0 * Wi + x1);
    const float v10 = __ldg(src + y1 * Wi + x0), v11 = __ldg(src + y1 * Wi + x1);
    const float v = (1.0f - ly) * ((1.0f - lx) * v00 + lx * v01) + ly * ((1.0f - lx) * v10 + lx * v11);
    if (!with_flip) {
      out[i] = v;
    } else {
      // planes of image b go to out images 2b (as is) and 2b+1 (mirrored): plane index b*C + c with C = 3
      const int64_t b = pl / 3, c = pl - b * 3;
      float* o0 = out + ((2 * b) * 3 + c) * (int64_t)So * So + (int64_t)oy * So;
      o0[ox] = v;
      o0[3 * (int64_t)So * So + (So - 1 - ox)] = v;
    }
  }
}

inline cudaError_t launch_resize_bilinear(const float* in, float* out, int batch, int Hi, int Wi, int So, int with_flip,
                                          cudaStream_t st) {
  const int64_t total = (int64_t)batch * 3 * So * So;
  if (total <= 0) return cudaSuccess;
  int64_t blocks = std::min<int64_t>((total + 255) / 256, (int64_t)kNumSMs * 16);
  cudaError_t r = launch_pdl(resize_bilinear_kernel, dim3((unsigned)blocks), dim3(256), 0, st, in, out, batch * 3, Hi, Wi,
                             So, with_flip);
  YNB_COUNT_LAUNCH();
  return r;
}

// =====================================================================================
// Pre-processing (SURVEY §8f row 1): the tail of data/transforms.py ValTransforms on the device.
//   Normalize (:59-70): x = float32(u8); x /= 255; x -= mean[c]; x /= std[c]   (c in BGR order)
//   ToTensor  (:394-398): BGR -> RGB, HWC -> CHW
//   Resize    (:73-119): pixels outside the letterboxed content carry the value mean*255
// in : uint8 [B,S,S,3] BGR, already resized / letterboxed to S x S on the host (cv2.resize stays there)
// out: float32 [B,3,S,S] RGB — what the stem reads.
// The normalisation is a pure function of (byte, channel): a 3 x 256 table computed on the host
// with the reference's exact float32 sequence, so the device result is bit-identical by
// construction.  4 pixels per thread: three 4-byte loads, three 16-byte stores.
// =====================================================================================
struct PreLut {
  float v[3][256];   // [input channel (B,G,R)][byte]
  float pad[3];      // normalised padding value per input channel
};

constexpr int kPreRows = 8;    // image rows per CTA (amortises the table load)

__global__ void __launch_bounds__(128)
preprocess_u8_kernel(const uint8_t* __restrict__ img, const int32_t* __restrict__ rects, float* __restrict__ out,
                     const PreLut* __restrict__ lut, int S) {
  __shared__ float s_lut[3][256];
  __shared__ float s_pad[3];
  pdl_trigger();
  const float* lg = &lut->v[0][0];
  for (int i = threadIdx.x; i < 768; i += 128) (&s_lut[0][0])[i] = __ldg(lg + i);   // coalesced, L2-resident
  if (threadIdx.x < 3) s_pad[threadIdx.x] = __ldg(&lut->pad[threadIdx.x]);
  pdl_wait();
  __syncthreads();
  const int x0 = (blockIdx.x * 128 + threadIdx.x) * 4;
  if (x0 >= S) return;
  const int b = blockIdx.z;
  int rx = 0, ry = 0, rw = S, rh = S;
  if (rects) { rx = rects[4 * b]; ry = rects[4 * b + 1]; rw = rects[4 * b + 2]; rh = rects[4 * b + 3]; }
#pragma unroll 2
  for (int y = blockIdx.y * kPreRows; y < min(S, (int)(blockIdx.y + 1) * kPreRows); ++y) {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(img + ((size_t)((size_t)b * S + y) * S + x0) * 3);
    const uint32_t w0 = __ldg(src), w1 = __ldg(src + 1), w2 = __ldg(src + 2);
    const bool row_in = y >= ry && y < ry + rh;
#pragma unroll
    for (int oc = 0; oc < 3; ++oc) {
      const int ic = 2 - oc;                            // RGB output plane <- BGR input channel
      float r[4];
#pragma unroll
      for (int px = 0; px < 4; ++px) {
        const int byte_idx = 3 * px + ic;               // 0..11 inside the three words
        const uint32_t word = byte_idx < 4 ? w0 : (byte_idx < 8 ? w1 : w2);
        const uint32_t v = (word >> ((byte_idx & 3) * 8)) & 0xffu;
        const bool in = row_in && x0 + px >= rx && x0 + px < rx + rw;
        r[px] = in ? s_lut[ic][v] : s_pad[ic];
      }
      *reinterpret_cast<float4*>(out + (((size_t)b * 3 + oc) * S + y) * S + x0) = make_float4(r[0], r[1], r[2], r[3]);
    }
  }
}

inline void make_prelut(PreLut* lut, const float mean_bgr[3], const float std_bgr[3]) {
  for (int c = 0; c < 3; ++c) {
    for (int v = 0; v < 256; ++v) {
      volatile float f = (float)v;      // volatile: every step rounds to float32, as the NumPy in-place ops do
      f = f / 255.0f;
      f = f - mean_bgr[c];
      f = f / std_bgr[c];
      lut->v[c][v] = f;
    }
    volatile float f = mean_bgr[c] * 255.0f;          // Resize.mean = [v * 255 for v in mean] (float32)
    f = f / 255.0f;
    f = f - mean_bgr[c];
    f = f / std_bgr[c];
    lut->pad[c] = f;
  }
}

// lut: DEVICE copy of the table
inline cudaError_t launch_preprocess_u8(const uint8_t* img, const int32_t* rects, float* out, const PreLut* lut,
                                        int batch, int S, cudaStream_t st) {
  if (batch <= 0) return cudaSuccess;
  if ((S & 3) || (reinterpret_cast<uintptr_t>(img) & 3u) || (reinterpret_cast<uintptr_t>(out) & 15u))
    return cudaErrorInvalidValue;
  dim3 grid((unsigned)((S / 4 + 127) / 128), (unsigned)((S + kPreRows - 1) / kPreRows), (unsigned)batch);
  cudaError_t r = launch_pdl(preprocess_u8_kernel, grid, dim3(128), 0, st, img, rects, out, lut, S);
  YNB_COUNT_LAUNCH();
  return r;
}

// =====================================================================================
// Whole ValTransforms on the device (SURVEY §8f row 1; data/transforms.py:73-119, 59-70, 394-398, 445-458):
// letterbox Resize (cv2.resize bilinear of the uint8 image + padding with mean*255) + Normalize + ToTensor, from
// the ORIGINAL uint8 BGR images (any shapes, packed in one buffer) straight to the float32 NCHW tensor the stem
// reads — the resized canvas never exists.  The bilinear resize restates OpenCV's 8-bit INTER_LINEAR exactly
// (imgproc/src/resize.cpp): float32 source coordinate, 11-bit fixed-point weights (cvRound), int32 horizontal
// pass, `(((b0 * (S0 >> 4)) >> 16) + ((b1 * (S1 >> 4)) >> 16) + 2) >> 2` vertically; exact 2x downscale = 2x2 mean.
// One thread per canvas pixel (three planes written, coalesced along x).
// =====================================================================================
struct ImageDesc {          // = ynb_image_desc of the C ABI
  long long offset;         // byte offset of the h0 x w0 x 3 uint8 image in the source buffer
  int h0, w0;               // source size
  int nw, nh;               // content size on the canvas
  int left, top;            // content position
  int mode;                 // 0: copy, 1: bilinear, 2: exact 2x2 area
  int pad_;
  double scale_x, scale_y;  // 1 / (nw / w0), 1 / (nh / h0) in float64, as cv::resize computes them
};

__device__ __forceinline__ void linear_coeff(int d, double scale, int sn, bool clamp_x, int* s0, int* s1, int* c0, int* c1) {
  const float f0 = (float)__dsub_rn(__dmul_rn(__dadd_rn((double)d, 0.5), scale), 0.5);
  int s = (int)floorf(f0);
  float f = __fsub_rn(f0, (float)s);
  if (clamp_x) {            // horizontal: out-of-range source columns get weight (1, 0) on the border column
    if (s < 0) { f = 0.0f; s = 0; }
    if (s >= sn - 1) { f = 0.0f; s = sn - 1; }
    *s0 = s; *s1 = min(s + 1, sn - 1);
  } else {                  // vertical: weights kept, rows clipped
    *s0 = min(max(s, 0), sn - 1); *s1 = min(max(s + 1, 0), sn - 1);
  }
  *c0 = __float2int_rn(__fmul_rn(__fsub_rn(1.0f, f), 2048.0f));
  *c1 = __float2int_rn(__fmul_rn(f, 2048.0f));
}

__global__ void __launch_bounds__(256)
letterbox_preprocess_kernel(const uint8_t* __restrict__ src, const ImageDesc* __restrict__ descs, float* __restrict__ out,
                            const PreLut* __restrict__ lut, int S) {
  __shared__ float s_lut[3][256];
  __shared__ float s_pad[3];
  const float* lg = &lut->v[0][0];
  for (int i = threadIdx.x; i < 768; i += 256) (&s_lut[0][0])[i] = __ldg(lg + i);
  if (threadIdx.x < 3) s_pad[threadIdx.x] = __ldg(&lut->pad[threadIdx.x]);
  __syncthreads();
  const int b = blockIdx.z, y = blockIdx.y;
  const int x = blockIdx.x * 256 + threadIdx.x;
  if (x >= S) return;
  const ImageDesc d = descs[b];
  const int dx = x - d.left, dy = y - d.top;
  float r[3];
  if (dx >= 0 && dx < d.nw && dy >= 0 && dy < d.nh) {
    const uint8_t* img = src + d.offset;
    const size_t pitch = (size_t)d.w0 * 3;
    int v[3];
    if (d.mode == 0) {
      const uint8_t* p = img + (size_t)dy * pitch + (size_t)dx * 3;
      v[0] = p[0]; v[1] = p[1]; v[2] = p[2];
    } else if (d.mode == 2) {
      const uint8_t* p = img + (size_t)(2 * dy) * pitch + (size_t)(2 * dx) * 3;
#pragma unroll
      for (int c = 0; c < 3; ++c) v[c] = ((int)p[c] + p[3 + c] + p[pitch + c] + p[pitch + 3 + c] + 2) >> 2;
    } else {
      int x0, x1, a0, a1, y0, y1, b0, b1;
      linear_coeff(dx, d.scale_x, d.w0, true, &x0, &x1, &a0, &a1);
      linear_coeff(dy, d.scale_y, d.h0, false, &y0, &y1, &b0, &b1);
      const uint8_t* r0 = img + (size_t)y0 * pitch;
      const uint8_t* r1 = img + (size_t)y1 * pitch;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const int h0v = (int)r0[x0 * 3 + c] * a0 + (int)r0[x1 * 3 + c] * a1;
        const int h1v = (int)r1[x0 * 3 + c] * a0 + (int)r1[x1 * 3 + c] * a1;
        v[c] = (((b0 * (h0v >> 4)) >> 16) + ((b1 * (h1v >> 4)) >> 16) + 2) >> 2;
      }
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) r[c] = s_lut[c][min(max(v[c], 0), 255)];
  } else {
#pragma unroll
    for (int c = 0; c < 3; ++c) r[c] = s_pad[c];
  }
#pragma unroll
  for (int oc = 0; oc < 3; ++oc)      // RGB output plane <- BGR input channel
    out[(((size_t)b * 3 + oc) * S + y) * S + x] = r[2 - oc];
}

inline cudaError_t launch_letterbox_preprocess(const uint8_t* src, const ImageDesc* descs, float* out, const PreLut* lut,
                                               int batch, int S, cudaStream_t st) {
  if (batch <= 0) return cudaSuccess;
  dim3 grid((unsigned)((S + 255) / 256), (unsigned)S, (unsigned)batch);
  letterbox_preprocess_kernel<<<grid, 256, 0, st>>>(src, descs, out, lut, S);
  YNB_COUNT_LAUNCH();
  return cudaGetLastError();
}

// Inverse box mapping of the evaluators (evaluator/cocoapi_evaluator.py:85-87, test.py:133-135) on the NMS output:
//   bboxes -= offset; bboxes /= scale; bboxes *= size      float32 array, float64 operands: each op in double,
// rounded to float32.  maps [B][12] = offset[4], scale[4], size[4]; rows [0, counts[b]) of image b.
__global__ void __launch_bounds__(256)
map_boxes_kernel(float* __restrict__ boxes, const int* __restrict__ counts, const double* __restrict__ maps, int batch,
                 long long n_per_image) {
  const int b = blockIdx.y;
  const double* m = maps + (size_t)b * 12;
  const long long total = (long long)min((long long)counts[b], n_per_image) * 4;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(i & 3);
    float* p = boxes + (size_t)b * n_per_image * 4 + i;
    float v = *p;
    v = (float)__dsub_rn((double)v, m[k]);
    v = (float)__ddiv_rn((double)v, m[4 + k]);
    v = (float)__dmul_rn((double)v, m[8 + k]);
    *p = v;
  }
}

inline cudaError_t launch_map_boxes(float* boxes, const int* counts, const double* maps, int batch, long long n_per_image,
                                    cudaStream_t st) {
  if (batch <= 0 || n_per_image <= 0) return cudaSuccess;
  const unsigned bx = (unsigned)std::min<long long>((n_per_image * 4 + 255) / 256, 64);
  map_boxes_kernel<<<dim3(bx, (unsigned)batch), 256, 0, st>>>(boxes, counts, maps, batch, n_per_image);
  YNB_COUNT_LAUNCH();
  return cudaGetLastError();
}

// =====================================================================================
// Depthwise 3x3, pad 1, stride 1|2, + bias (+ activation).  NHWC, 4 channels per thread
// with 16-byte loads; consecutive threads take consecutive channel groups of one pixel,
// so a warp reads whole 128-byte lines.  (backbone/shufflenetv2.py:66-67; heads
// models/yolo_nano.py:51,53)
//   w [9][C4] tap-major, b [C4]  (C4 = channels rounded to 4; pads are zero)
// =====================================================================================
// Each thread produces kDwTX consecutive output pixels of one 4-channel group: the 3 x
// ((TX-1)*stride+3) input window is loaded once into registers (4.5 instead of 9 16-byte
// loads per output at stride 1) and the 9 filter taps once per thread, which takes the
// kernel off the L1 bandwidth limit the one-pixel-per-thread version sat on.
constexpr int kDwTX = 4;

constexpr int kDwThreads = 128;

// grid: x = ceil(channel groups * x groups / 128), y = output row, z = image — the only index
// arithmetic left per thread is one division; all addressing inside an image is 32-bit.
template <int STRIDE>
__global__ void __launch_bounds__(kDwThreads)
dwconv3x3_kernel(const float* __restrict__ in, int in_ld, int in_off,
                 float* __restrict__ out, int out_ld, int out_off,
                 const float* __restrict__ w, const float* __restrict__ bias,
                 int Hin, int Win, int Ho, int Wo, int groups, int xgroups, int C4, int act) {
  constexpr int NIN = (kDwTX - 1) * STRIDE + 3;
  pdl_trigger();
  const int t = blockIdx.x * kDwThreads + threadIdx.x;
  if (t >= groups * xgroups) { pdl_wait(); return; }
  const int xg = t / groups, g = t - xg * groups;
  const int yo = blockIdx.y, b = blockIdx.z;
  const int c = g << 2;
  const int xo0 = xg * kDwTX;
  const float4 bv = __ldg(reinterpret_cast<const float4*>(bias + c));
  float4 kw[9];
#pragma unroll
  for (int k = 0; k < 9; ++k) kw[k] = __ldg(reinterpret_cast<const float4*>(w + k * C4 + c));
  pdl_wait();
  float4 acc[kDwTX];
#pragma unroll
  for (int q = 0; q < kDwTX; ++q) acc[q] = bv;
  const float* inb = in + (size_t)b * Hin * Win * in_ld + in_off + c;
  const int xi0 = xo0 * STRIDE - 1;
#pragma unroll
  for (int ky = 0; ky < 3; ++ky) {
    const int yi = yo * STRIDE + ky - 1;
    if (yi < 0 || yi >= Hin) continue;
    const float* rowp = inb + (yi * Win + xi0) * in_ld;          // 32-bit offsets inside an image
    float4 v[NIN];
#pragma unroll
    for (int j = 0; j < NIN; ++j) {
      const int xi = xi0 + j;
      v[j] = (xi >= 0 && xi < Win) ? __ldg(reinterpret_cast<const float4*>(rowp + j * in_ld))
                                   : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int kx = 0; kx < 3; ++kx) {
      const float4 k = kw[ky * 3 + kx];
#pragma unroll
      for (int q = 0; q < kDwTX; ++q) {
        const float4 u = v[q * STRIDE + kx];
        // packed FFMA2: two fp32 FMAs per issue slot, each rounded like fmaf
        const float2 lo = __ffma2_rn(make_float2(u.x, u.y), make_float2(k.x, k.y), make_float2(acc[q].x, acc[q].y));
        const float2 hi = __ffma2_rn(make_float2(u.z, u.w), make_float2(k.z, k.w), make_float2(acc[q].z, acc[q].w));
        acc[q] = make_float4(lo.x, lo.y, hi.x, hi.y);
      }
    }
  }
  float* ob = out + (size_t)b * Ho * Wo * out_ld + (yo * Wo + xo0) * out_ld + out_off + c;
#pragma unroll
  for (int q = 0; q < kDwTX; ++q) {
    if (xo0 + q < Wo) {
      float4 a = acc[q];
      a.x = apply_act(a.x, act); a.y = apply_act(a.y, act); a.z = apply_act(a.z, act); a.w = apply_act(a.w, act);
      *reinterpret_cast<float4*>(ob + q * out_ld) = a;
    }
  }
}

// ---- TMA-tiled variant (the product path) -----------------------------------------------------
// One CTA = one spatial tile x one 32-channel chunk x one image.  The input tile WITH ITS HALO arrives
// as a single 4-D TMA box ([32 ch] x IW x IH pixels, 128-byte swizzle); pixels outside the image are
// zero-filled by the copy engine (= the conv's zero padding), channels beyond the view likewise.  A
// thread then computes a 1x4 strip of outputs for one 4-channel group from shared memory: no bounds
// checks, no address arithmetic per tap — ~5x fewer instructions per output than the register-tiled
// global-load kernel above, which stays as the fallback for unaligned views.
template <int STRIDE, typename E = float>
struct DwTile {
  static constexpr int TW = STRIDE == 1 ? 16 : 8;      // outputs per tile
  static constexpr int TH = 8;
  static constexpr int IW = (TW - 1) * STRIDE + 3;     // 18 | 17 input pixels with halo
  static constexpr int IH = (TH - 1) * STRIDE + 3;     // 10 | 17
  static constexpr int CGS = 32 / sizeof(E);           // 4-channel groups per 128-byte pixel row: 8 (float) | 16 (bf16)
  static constexpr int CHUNK = CGS * 4;                // channels per CTA: 32 | 64
  static constexpr int THREADS = (TW / 4) * TH * CGS;  // strips x channel groups: 256 | 128 (float), 512 | 256 (bf16)
  static constexpr int BYTES = IW * IH * 128;
};

// REV: taps reversed and no bias = the gradient of a stride-1 depthwise conv w.r.t. its input
// (train_ops.cuh / ynb_dwconv3x3_bwd_data).
template <int STRIDE, bool REV = false, typename E = float>
__global__ void __launch_bounds__(DwTile<STRIDE, E>::THREADS)
dwconv3x3_tma_kernel(const __grid_constant__ CUtensorMap tmIn, E* __restrict__ out, int out_ld, int out_off,
                     const float* __restrict__ w, const float* __restrict__ bias, int Ho, int Wo, int C4,
                     int tiles_x, int act) {
  using T = DwTile<STRIDE, E>;
  __shared__ __align__(1024) uint8_t s_tile[T::BYTES];
  __shared__ __align__(8) uint64_t s_bar;
  const int tid = threadIdx.x;
  const int ty = blockIdx.x / tiles_x, tx = blockIdx.x - ty * tiles_x;
  const int chunk = blockIdx.y, b = blockIdx.z;
  const int x0 = tx * T::TW, y0 = ty * T::TH;
  pdl_trigger();
  if (tid == 0) {
    ptx::mbar_init(&s_bar, 1);
    ptx::fence_barrier_init();
  }
  // weights of this thread's 4 channels (independent of the previous kernel)
  const int cg = tid & (T::CGS - 1);                    // 4-channel group inside the chunk
  const int c = chunk * T::CHUNK + cg * 4;
  const bool c_ok = c < C4;
  float4 kw[9], bv = make_float4(0.f, 0.f, 0.f, 0.f);
  if (c_ok) {
    if (!REV) bv = __ldg(reinterpret_cast<const float4*>(bias + c));
#pragma unroll
    for (int k = 0; k < 9; ++k) kw[k] = __ldg(reinterpret_cast<const float4*>(w + (REV ? 8 - k : k) * C4 + c));
  }
  pdl_wait();
  if (tid == 0) {
    ptx::mbar_arrive_expect_tx(&s_bar, T::BYTES);
    ptx::tma_load_4d(s_tile, &tmIn, &s_bar, chunk * T::CHUNK, x0 * STRIDE - 1, y0 * STRIDE - 1, b);
  }
  __syncthreads();                                      // barrier init visible
  ptx::mbar_wait(&s_bar, 0, nullptr, 0);
  if (!c_ok) return;
  const int strip = tid / T::CGS;                       // (sy, sx): 4 outputs along x
  const int sy = strip / (T::TW / 4), sx = strip - sy * (T::TW / 4);
  const int yo = y0 + sy, xo = x0 + sx * 4;
  if (yo >= Ho || xo >= Wo) return;
  constexpr int NIN = 3 * STRIDE + 3;                   // input columns feeding 4 outputs: 6 | 9
  float4 acc[4] = {bv, bv, bv, bv};
#pragma unroll
  for (int ky = 0; ky < 3; ++ky) {
    const int r0 = (sy * STRIDE + ky) * T::IW + sx * 4 * STRIDE;      // first pixel row of the tile buffer
    float4 v[NIN];
#pragma unroll
    for (int j = 0; j < NIN; ++j) {
      const int r = r0 + j;
      // 128-byte swizzle: 16-byte chunk index ^ (row & 7); a 4-channel group is a whole chunk (float) or half of one (bf16)
      if (sizeof(E) == 4) v[j] = load4(reinterpret_cast<const E*>(s_tile + r * 128 + ((cg ^ (r & 7)) << 4)));
      else v[j] = load4(reinterpret_cast<const E*>(s_tile + r * 128 + ((((cg >> 1) ^ (r & 7)) << 4) | ((cg & 1) << 3))));
    }
#pragma unroll
    for (int kx = 0; kx < 3; ++kx) {
      const float4 k = kw[ky * 3 + kx];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float4 u = v[q * STRIDE + kx];
        const float2 lo = __ffma2_rn(make_float2(u.x, u.y), make_float2(k.x, k.y), make_float2(acc[q].x, acc[q].y));
        const float2 hi = __ffma2_rn(make_float2(u.z, u.w), make_float2(k.z, k.w), make_float2(acc[q].z, acc[q].w));
        acc[q] = make_float4(lo.x, lo.y, hi.x, hi.y);
      }
    }
  }
  E* ob = out + (size_t)b * Ho * Wo * out_ld + (yo * Wo + xo) * out_ld + out_off + c;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    if (xo + q < Wo) {
      float4 a = acc[q];
      a.x = apply_act(a.x, act); a.y = apply_act(a.y, act); a.z = apply_act(a.z, act); a.w = apply_act(a.w, act);
      store4(ob + q * out_ld, a);
    }
  }
}

// tensor map over the input view [B][Hin][Win][C4 of ld]: boxes of 128 bytes of channels x IW x IH pixels
inline bool make_tmap_dw(CUtensorMap* m, const void* in, int in_ld, int in_off, int batch, int Hin, int Win, int C4,
                         int stride, bool is_bf16 = false) {
  const int es = is_bf16 ? 2 : 4;
  const char* base = static_cast<const char*>(in) + (size_t)in_off * es;
  if ((reinterpret_cast<uintptr_t>(base) & 15u) || ((in_ld * es) & 15)) return false;
  return stride == 1 ? make_tmap_nhwc(m, base, C4, Win, Hin, batch, in_ld, DwTile<1>::IW, DwTile<1>::IH, is_bf16)
                     : make_tmap_nhwc(m, base, C4, Win, Hin, batch, in_ld, DwTile<2>::IW, DwTile<2>::IH, is_bf16);
}

template <typename E>
inline cudaError_t launch_dwconv3x3_tma_t(const CUtensorMap& tm, E* out, int out_ld, int out_off, const float* w,
                                          const float* b, int batch, int Hin, int Win, int C4, int stride, int act,
                                          cudaStream_t st, bool reversed_taps) {
  const int Ho = (Hin - 1) / stride + 1, Wo = (Win - 1) / stride + 1;
  if (batch <= 0 || C4 <= 0) return cudaSuccess;
  const int TW = stride == 1 ? DwTile<1>::TW : DwTile<2>::TW, TH = DwTile<1>::TH;
  const int tiles_x = (Wo + TW - 1) / TW, tiles_y = (Ho + TH - 1) / TH;
  constexpr int CH = DwTile<1, E>::CHUNK;
  dim3 grid((unsigned)(tiles_x * tiles_y), (unsigned)((C4 + CH - 1) / CH), (unsigned)batch);
  if (reversed_taps) {
    if (stride != 1) return cudaErrorInvalidValue;
    cudaError_t rr = launch_pdl(dwconv3x3_tma_kernel<1, true, E>, grid, dim3(DwTile<1, E>::THREADS), 0, st, tm, out, out_ld,
                                out_off, w, b, Ho, Wo, C4, tiles_x, act);
    YNB_COUNT_LAUNCH();
    return rr;
  }
  cudaError_t r = stride == 1
      ? launch_pdl(dwconv3x3_tma_kernel<1, false, E>, grid, dim3(DwTile<1, E>::THREADS), 0, st, tm, out, out_ld, out_off, w,
                   b, Ho, Wo, C4, tiles_x, act)
      : launch_pdl(dwconv3x3_tma_kernel<2, false, E>, grid, dim3(DwTile<2, E>::THREADS), 0, st, tm, out, out_ld, out_off, w,
                   b, Ho, Wo, C4, tiles_x, act);
  YNB_COUNT_LAUNCH();
  return r;
}

inline cudaError_t launch_dwconv3x3_tma(const CUtensorMap& tm, void* out, int out_ld, int out_off, const float* w,
                                        const float* b, int batch, int Hin, int Win, int C4, int stride, int act,
                                        cudaStream_t st, bool reversed_taps = false, bool is_bf16 = false) {
  return is_bf16 ? launch_dwconv3x3_tma_t(tm, static_cast<bf16*>(out), out_ld, out_off, w, b, batch, Hin, Win, C4, stride,
                                          act, st, reversed_taps)
                 : launch_dwconv3x3_tma_t(tm, static_cast<float*>(out), out_ld, out_off, w, b, batch, Hin, Win, C4, stride,
                                          act, st, reversed_taps);
}

inline cudaError_t launch_dwconv3x3(const float* in, int in_ld, int in_off, float* out, int out_ld,
                                    int out_off, const float* w, const float* b, int batch, int Hin,
                                    int Win, int C4, int stride, int act, cudaStream_t st) {
  const int Ho = (Hin - 1) / stride + 1, Wo = (Win - 1) / stride + 1;
  const int groups = C4 / 4, xgroups = (Wo + kDwTX - 1) / kDwTX;
  if (batch <= 0 || Ho <= 0 || groups <= 0) return cudaSuccess;
  if (Ho > 65535 || batch > 65535) return cudaErrorInvalidValue;
  dim3 grid((unsigned)((groups * xgroups + kDwThreads - 1) / kDwThreads), (unsigned)Ho, (unsigned)batch);
  cudaError_t r = launch_pdl(stride == 1 ? dwconv3x3_kernel<1> : dwconv3x3_kernel<2>, grid, dim3(kDwThreads), 0, st, in,
                             in_ld, in_off, out, out_ld, out_off, w, b, Hin, Win, Ho, Wo, groups, xgroups, C4, act);
  YNB_COUNT_LAUNCH();
  return r;
}

// =====================================================================================
// Pass-through half of a stride-1 ShuffleNetV2 unit: out[m, 2i] = in[m, i], i < half.
// Together with the branch-2 epilogue (which writes channel 2i+1) this IS
// torch.cat + channel_shuffle (backbone/shufflenetv2.py:70-76, 14-28): no shuffle copy.
// =====================================================================================
__global__ void __launch_bounds__(256)
interleave_copy_kernel(const float* __restrict__ in, int in_ld, float* __restrict__ out, int out_ld,
                       int64_t pixels, int half) {
  const int64_t total = pixels * half;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    int c = (int)(i % half);
    int64_t m = i / half;
    out[m * out_ld + 2 * c] = __ldg(in + m * in_ld + c);
  }
}

inline cudaError_t launch_interleave_copy(const float* in, int in_ld, float* out, int out_ld,
                                          int64_t pixels, int half, cudaStream_t st) {
  int64_t blocks = (pixels * half + 255) / 256;
  int64_t cap = (int64_t)kNumSMs * 16;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  interleave_copy_kernel<<<(unsigned)blocks, 256, 0, st>>>(in, in_ld, out, out_ld, pixels, half);
  YNB_COUNT_LAUNCH();
  return cudaGetLastError();
}

// =====================================================================================
// Tap / parity hook: internal NHWC -> canonical NCHW.
// Tiled transpose through shared memory: coalesced on both sides.
// =====================================================================================
template <typename E>
__global__ void __launch_bounds__(256)
nhwc_to_nchw_kernel(const E* __restrict__ in, int in_ld, float* __restrict__ out,
                    int C, int HW) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z;
  const int p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 32 x 8
  for (int r = ty; r < 32; r += 8) {
    int p = p0 + r, c = c0 + tx;
    float v = 0.0f;
    if (p < HW && c < C) v = to_float(in[((size_t)b * HW + p) * in_ld + c]);
    tile[r][tx] = v;
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    int c = c0 + r, p = p0 + tx;
    if (p < HW && c < C) out[((size_t)b * C + c) * HW + p] = tile[tx][r];
  }
}

inline cudaError_t launch_nhwc_to_nchw(const void* in, int in_ld, float* out,
                                       int batch, int C, int HW, cudaStream_t st, bool in_bf16 = false) {
  dim3 grid((HW + 31) / 32, (C + 31) / 32, batch);
  if (in_bf16) nhwc_to_nchw_kernel<<<grid, 256, 0, st>>>(static_cast<const bf16*>(in), in_ld, out, C, HW);
  else nhwc_to_nchw_kernel<<<grid, 256, 0, st>>>(static_cast<const float*>(in), in_ld, out, C, HW);
  YNB_COUNT_LAUNCH();
  return cudaGetLastError();
}

// =====================================================================================
// FPN / PAN merge: out = a + nearest_resample(a2)   (models/yolo_nano.py:291-296;
// F.interpolate default mode 'nearest': up x2 replicates pixels, x0.5 takes [::2, ::2]).
// mode 1: a2 is (H/2 x W/2), mode 2: a2 is (2H x 2W).  All tensors share `ld` = 96.
// =====================================================================================
__device__ __forceinline__ float tf32_rn(float x) {     // same bits as rn_tf32_bits() of gemm_tc.cuh
  return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u);
}

template <typename E>
__global__ void __launch_bounds__(256)
resample_add_kernel(const E* __restrict__ a, const E* __restrict__ a2, E* __restrict__ out,
                    E* __restrict__ out_lo, int batch, int H, int W, int ld, int mode) {
  const int groups = ld >> 2;
  const int64_t total = (int64_t)batch * H * W * groups;
  const int H2 = mode == 1 ? H >> 1 : H << 1, W2 = mode == 1 ? W >> 1 : W << 1;
  pdl_trigger();
  pdl_wait();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    int g = (int)(i % groups);
    int64_t p = i / groups;
    int x = (int)(p % W);
    int y = (int)((p / W) % H);
    int b = (int)(p / ((int64_t)W * H));
    int y2 = mode == 1 ? y >> 1 : y << 1, x2 = mode == 1 ? x >> 1 : x << 1;
    float4 u = load4(a + p * ld + 4 * g);
    float4 v = load4(a2 + (((size_t)b * H2 + y2) * W2 + x2) * ld + 4 * g);
    u.x += v.x; u.y += v.y; u.z += v.z; u.w += v.w;
    if (sizeof(E) == 4 && out_lo != nullptr) {
      // The sum feeds a 3x3 conv on the tensor cores in fp32-parity mode: every element would be
      // split into exact-tf32 hi + lo nine times (once per tap) inside the GEMM.  Split it ONCE here
      // (round to nearest, as the GEMM's splitters do) and let the GEMM load both planes.
      float4 h, l;
      h.x = tf32_rn(u.x); h.y = tf32_rn(u.y); h.z = tf32_rn(u.z); h.w = tf32_rn(u.w);
      l.x = tf32_rn(u.x - h.x); l.y = tf32_rn(u.y - h.y); l.z = tf32_rn(u.z - h.z); l.w = tf32_rn(u.w - h.w);
      store4(out + p * ld + 4 * g, h);
      store4(out_lo + p * ld + 4 * g, l);
    } else {
      store4(out + p * ld + 4 * g, u);
    }
  }
}

inline cudaError_t launch_resample_add(const void* a, const void* a2, void* out, void* out_lo, int batch, int H,
                                       int W, int ld, int mode, cudaStream_t st, bool is_bf16 = false) {
  int64_t total = (int64_t)batch * H * W * (ld / 4);
  int64_t blocks = (total + 255) / 256;
  int64_t cap = (int64_t)kNumSMs * 16;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  cudaError_t r = is_bf16
      ? launch_pdl(resample_add_kernel<bf16>, dim3((unsigned)blocks), dim3(256), 0, st, static_cast<const bf16*>(a),
                   static_cast<const bf16*>(a2), static_cast<bf16*>(out), static_cast<bf16*>(nullptr), batch, H, W, ld, mode)
      : launch_pdl(resample_add_kernel<float>, dim3((unsigned)blocks), dim3(256), 0, st, static_cast<const float*>(a),
                   static_cast<const float*>(a2), static_cast<float*>(out), static_cast<float*>(out_lo), batch, H, W, ld, mode);
  YNB_COUNT_LAUNCH();
  return r;
}

}  // namespace ynb
