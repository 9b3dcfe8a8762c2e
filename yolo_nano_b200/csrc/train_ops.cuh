// Training branch at the head boundary (SURVEY §8 row a14, §8f row 4): target assignment, the four
// losses with their gradient w.r.t. the raw head maps, the SGD update, and the backward kernels of
// the depthwise / pointwise convolutions.  All HBM-bound streaming kernels: coalesced row access,
// grids sized in multiples of the SM count, deterministic two-stage reductions (no float atomics).
#pragma once
#include "common.cuh"

namespace ynb {

constexpr int kTrainMaxAnchors = 8;
constexpr int kLossThreads = 256;
constexpr int kLossCells = 64;                // cells (pixels of one level of one image) per block

struct TrainLossParams {
  const float* raw[3];     // NHWC [B, HW_l, ld], channel map obj a | cls A + a*C + c | box A(1+C) + 4a + k
  float* grad[3];          // same layout: d(conf + cls + bbox + iou loss) / d raw
  const float* target;     // [B, N, 11]  (tools.py:97-216)
  double* partials;        // [gridDim.x][4]
  int ld, B, A, C, S;
  int grid[3], stride[3];
  int cells[3];            // HW_l
  int cell_off[3];         // prefix of cells
  int tiles[3];            // ceil(HW_l / kLossCells)
  int tiles_per_image;
  int cells_total;         // sum HW_l
  float anchors[3][kTrainMaxAnchors][2];
};

__device__ __forceinline__ float sigmoid_precise(float v) { return 1.0f / (1.0f + expf(-v)); }
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// One block per tile of 64 cells of one level of one image (= 64 contiguous rows of the raw map and
// 64*A contiguous target rows).
//   phase 0: the tile's targets (64*A*11 floats, contiguous) are staged in shared memory, coalesced;
//   phase 1: one thread per anchor does the scalar work — decode, IoU, objectness / box / IoU losses
//            and their gradients (5 floats per anchor -> shared memory);
//   phase 2: all threads write the 64 gradient rows ONCE with 16-byte stores: objectness and box
//            columns from shared memory, zeros in the class columns (their gradient is zero for every
//            non-positive anchor, so the class logits of those are never read);
//   phase 3: one warp per positive anchor: cross entropy and the softmax gradient of its C
//            class columns.
// HBM traffic = obj/box logits + targets + the gradient map written once (+ C logits per positive).
//   models/yolo_nano.py:333-358: decode (no clamp) -> iou_score -> gt_conf = iou (detached)
//   tools.py:12-34   MSEWithLogitsLoss: 5*pos*(sigmoid(l) - iou)^2 + neg*sigmoid(l)^2
//   tools.py:236-276 CE on positives, BCE-with-logits (txty) and MSE (twth) weighted by
//                    gt_box_scale_weight*mask, SmoothL1(iou, mask) over ALL anchors; each sum / B.
__global__ void __launch_bounds__(kLossThreads) train_loss_kernel(const TrainLossParams p) {
  extern __shared__ __align__(16) float sh_dyn[];
  const int A = p.A, C = p.C;
  float* sh_t = sh_dyn;                                   // [64*A][11] targets
  float* sh_g = sh_t + kLossCells * A * 11;               // [64*A][5] g_conf, g_tx, g_ty, g_tw, g_th
  __shared__ double part[kLossThreads / 32][4];

  const int b = blockIdx.x / p.tiles_per_image;
  int tile = blockIdx.x - b * p.tiles_per_image;
  int lvl = 0;
  if (tile >= p.tiles[0]) { tile -= p.tiles[0]; lvl = 1; }
  if (lvl == 1 && tile >= p.tiles[1]) { tile -= p.tiles[1]; lvl = 2; }
  const int cell0 = tile * kLossCells;
  const int ncell = min(kLossCells, p.cells[lvl] - cell0);
  const int nanch = ncell * A;
  const int used = A * (1 + C + 4);
  const float invB = 1.0f / (float)p.B;
  const float fS = (float)p.S;
  const float fs = (float)p.stride[lvl];
  const long long N = (long long)p.cells_total * A;
  const float* __restrict__ raw = p.raw[lvl] + ((long long)b * p.cells[lvl] + cell0) * p.ld;
  float* __restrict__ g = p.grad[lvl] + ((long long)b * p.cells[lvl] + cell0) * p.ld;
  const float* __restrict__ tg = p.target + ((long long)b * N + ((long long)p.cell_off[lvl] + cell0) * A) * 11;

  for (int i = threadIdx.x; i < nanch * 11; i += kLossThreads) sh_t[i] = tg[i];
  __syncthreads();

  float l_conf = 0.0f, l_box = 0.0f, l_iou = 0.0f, l_cls = 0.0f;
  for (int i = threadIdx.x; i < nanch; i += kLossThreads) {      // one pass when 64*A <= 256
    const int cl = i / A, a = i - cl * A;
    const int cell = cell0 + cl;
    const int gy = cell / p.grid[lvl], gx = cell - gy * p.grid[lvl];
    const float* __restrict__ t = sh_t + i * 11;
    const float* __restrict__ row = raw + (long long)cl * p.ld;
    const float obj = t[0];
    const float mask = obj > 0.0f ? 1.0f : 0.0f;
    const float pos = obj == 1.0f ? 1.0f : 0.0f;
    const float neg = obj == 0.0f ? 1.0f : 0.0f;
    const float lconf = row[a];
    const int bo = A * (1 + C) + 4 * a;
    const float tx = row[bo], ty = row[bo + 1], tw = row[bo + 2], th = row[bo + 3];
    // decode_boxes / input_size (models/yolo_nano.py:120-156,337)
    const float sx = sigmoid_precise(tx), sy = sigmoid_precise(ty);
    const float ew = expf(tw), eh = expf(th);
    const float aw = p.anchors[lvl][a][0], ah = p.anchors[lvl][a][1];
    const float cx = __fmul_rn(__fadd_rn(sx, (float)gx), fs), cy = __fmul_rn(__fadd_rn(sy, (float)gy), fs);
    const float bw = __fmul_rn(ew, aw), bh = __fmul_rn(eh, ah);
    const float x1 = __fsub_rn(cx, bw * 0.5f) / fS, y1 = __fsub_rn(cy, bh * 0.5f) / fS;
    const float x2 = __fadd_rn(cx, bw * 0.5f) / fS, y2 = __fadd_rn(cy, bh * 0.5f) / fS;
    // iou_score (tools.py:219-233)
    const float q1x = t[7], q1y = t[8], q2x = t[9], q2y = t[10];
    const float tlx = fmaxf(x1, q1x), tly = fmaxf(y1, q1y), brx = fminf(x2, q2x), bry = fminf(y2, q2y);
    const float wa = __fsub_rn(x2, x1), ha = __fsub_rn(y2, y1);
    const float area_a = __fmul_rn(wa, ha);
    const float area_b = __fmul_rn(__fsub_rn(q2x, q1x), __fsub_rn(q2y, q1y));
    const float en = (tlx < brx && tly < bry) ? 1.0f : 0.0f;
    const float iw = __fsub_rn(brx, tlx), ih = __fsub_rn(bry, tly);
    const float area_i = __fmul_rn(__fmul_rn(iw, ih), en);
    const float uni = __fsub_rn(__fadd_rn(area_a, area_b), area_i);
    const float iou = area_i / uni;
    // objectness (tools.py:12-34); the label is the detached IoU
    const float pc = sigmoid_precise(lconf);
    const float dpi = pc - iou;
    l_conf += 5.0f * (pos * dpi * dpi) + neg * pc * pc;
    const float g_conf = (10.0f * pos * dpi + 2.0f * neg * pc) * pc * (1.0f - pc) * invB;
    // iou loss: SmoothL1(iou, mask), beta = 1 (tools.py:273)
    const float d = iou - mask, ad = fabsf(d);
    l_iou += ad < 1.0f ? 0.5f * d * d : ad - 0.5f;
    const float g_iou = (ad < 1.0f ? d : (d > 0.0f ? 1.0f : -1.0f)) * invB;
    // ... back through iou = I / (Aa + Ab - I)
    const float inv_u = 1.0f / uni;
    const float g_I = g_iou * (inv_u + area_i * inv_u * inv_u);
    const float g_Aa = -g_iou * area_i * inv_u * inv_u;
    const float g_iw = g_I * ih * en, g_ih = g_I * iw * en;
    // torch.max / torch.min of two tensors split the gradient evenly on ties
    const float sx2 = x2 < q2x ? 1.0f : (x2 == q2x ? 0.5f : 0.0f), sx1 = x1 > q1x ? 1.0f : (x1 == q1x ? 0.5f : 0.0f);
    const float sy2 = y2 < q2y ? 1.0f : (y2 == q2y ? 0.5f : 0.0f), sy1 = y1 > q1y ? 1.0f : (y1 == q1y ? 0.5f : 0.0f);
    const float g_x2 = (g_iw * sx2 + g_Aa * ha) / fS, g_x1 = (-g_iw * sx1 - g_Aa * ha) / fS;
    const float g_y2 = (g_ih * sy2 + g_Aa * wa) / fS, g_y1 = (-g_ih * sy1 - g_Aa * wa) / fS;
    float g_tx = (g_x1 + g_x2) * fs * sx * (1.0f - sx);
    float g_ty = (g_y1 + g_y2) * fs * sy * (1.0f - sy);
    float g_tw = (g_x2 - g_x1) * 0.5f * bw;
    float g_th = (g_y2 - g_y1) * 0.5f * bh;
    if (mask > 0.0f) {   // box loss (tools.py:267-270)
      const float wm = t[6];
      const float ttx = t[2], tty = t[3], ttw = t[4], tth = t[5];
      const float bce = (fmaxf(tx, 0.0f) - tx * ttx + log1pf(expf(-fabsf(tx)))) +
                        (fmaxf(ty, 0.0f) - ty * tty + log1pf(expf(-fabsf(ty))));
      const float mse = (tw - ttw) * (tw - ttw) + (th - tth) * (th - tth);
      l_box += bce * wm + mse * wm;
      g_tx += wm * (sx - ttx) * invB;
      g_ty += wm * (sy - tty) * invB;
      g_tw += wm * 2.0f * (tw - ttw) * invB;
      g_th += wm * 2.0f * (th - tth) * invB;
    }
    float* gq = sh_g + i * 5;
    gq[0] = g_conf; gq[1] = g_tx; gq[2] = g_ty; gq[3] = g_tw; gq[4] = g_th;
  }
  __syncthreads();

  // phase 2: the gradient rows, written once.  Column c of a row: c < A -> g_conf of anchor c;
  // c in [A(1+C), used) -> box gradient; everything else (class columns, padding) 0.
  const int box0 = A * (1 + C);
  if ((p.ld & 3) == 0) {
    // a warp per row, a lane per 16-byte column group: no index division, and the class-only groups
    // (59 of 64 at A = 3, C = 80) are stored as zeros without touching shared memory
    const int ld4 = p.ld >> 2;
    const int lane2 = threadIdx.x & 31, warp2 = threadIdx.x >> 5;
    for (int cl = warp2; cl < ncell; cl += kLossThreads / 32) {
      float4* grow4 = reinterpret_cast<float4*>(g + (long long)cl * p.ld);
      const float* gq = sh_g + cl * A * 5;
      for (int c4 = lane2; c4 < ld4; c4 += 32) {
        const int c = c4 << 2;
        float v[4] = {0.0f, 0.0f, 0.0f, 0.0f};
        if (c < A || c + 3 >= box0) {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int cc = c + k;
            if (cc < A) v[k] = gq[cc * 5];
            else if (cc >= box0 && cc < used) v[k] = gq[((cc - box0) >> 2) * 5 + 1 + ((cc - box0) & 3)];
          }
        }
        grow4[c4] = make_float4(v[0], v[1], v[2], v[3]);
      }
    }
  } else {
    for (int i = threadIdx.x; i < ncell * p.ld; i += kLossThreads) {
      const int cl = i / p.ld, cc = i - cl * p.ld;
      float val = 0.0f;
      if (cc < A) val = sh_g[(cl * A + cc) * 5];
      else if (cc >= box0 && cc < used) val = sh_g[(cl * A + ((cc - box0) >> 2)) * 5 + 1 + ((cc - box0) & 3)];
      g[(long long)cl * p.ld + cc] = val;
    }
  }
  __syncthreads();

  // phase 3: class loss of the positives: cross entropy (tools.py:264), one warp per positive.
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int i = warp; i < nanch; i += kLossThreads / 32) {      // fixed anchor -> warp map: deterministic sums
    if (!(sh_t[i * 11] > 0.0f)) continue;
    const int cl = i / A, a = i - cl * A;
    const float* __restrict__ row = raw + (long long)cl * p.ld + A + a * C;
    float* __restrict__ grow = g + (long long)cl * p.ld + A + a * C;
    const int gt = (int)sh_t[i * 11 + 1];
    float m = -INFINITY;
    for (int c = lane; c < C; c += 32) m = fmaxf(m, row[c]);
    m = warp_max(m);
    float s = 0.0f;
    for (int c = lane; c < C; c += 32) s += expf(row[c] - m);
    s = warp_sum(s);
    const float inv_s = 1.0f / s;
    for (int c = lane; c < C; c += 32) grow[c] = (expf(row[c] - m) * inv_s - (c == gt ? 1.0f : 0.0f)) * invB;
    if (lane == 0) l_cls += logf(s) + m - row[gt];
  }

  // block partial of the four sums (float per thread, double across threads; fixed order)
  float acc[4] = {l_conf, l_cls, l_box, l_iou};
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float wsum = warp_sum(acc[k]);
    if (lane == 0) part[warp][k] = (double)wsum;
  }
  __syncthreads();
  if (threadIdx.x < 4) {
    double s = 0.0;
    for (int w = 0; w < kLossThreads / 32; ++w) s += part[w][threadIdx.x];
    p.partials[(long long)blockIdx.x * 4 + threadIdx.x] = s;
  }
}

// Second stage: fixed-order sum of the block partials, / batch_size.  256 threads per loss keep the serial
// chain at blocks / 256 loads (a single warp per loss cost 9 us at 1824 blocks), then a fixed tree.
__global__ void __launch_bounds__(1024) train_loss_finalize_kernel(const double* __restrict__ partials, int blocks, int B,
                                                                   float* __restrict__ losses) {
  __shared__ double sh[4][256];
  const int k = threadIdx.x >> 8, i = threadIdx.x & 255;
  double s = 0.0;
  for (int j = i; j < blocks; j += 256) s += partials[(long long)j * 4 + k];
  sh[k][i] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (i < o) sh[k][i] += sh[k][i + o];
    __syncthreads();
  }
  if (i == 0) losses[k] = (float)(sh[k][0] / (double)B);
}

inline int train_loss_blocks(int batch, int input_size) {
  int tiles = 0;
  for (int s = 8; s <= 32; s *= 2) tiles += ((input_size / s) * (input_size / s) + kLossCells - 1) / kLossCells;
  return tiles * batch;
}

inline cudaError_t launch_train_loss(TrainLossParams p, float* losses, cudaStream_t st) {
  p.tiles_per_image = 0;
  for (int l = 0; l < 3; ++l) {
    p.tiles[l] = (p.cells[l] + kLossCells - 1) / kLossCells;
    p.tiles_per_image += p.tiles[l];
  }
  const int blocks = p.tiles_per_image * p.B;
  const size_t smem = (size_t)kLossCells * p.A * (11 + 5) * sizeof(float);
  train_loss_kernel<<<blocks, kLossThreads, smem, st>>>(p);
  YNB_COUNT_LAUNCH();
  train_loss_finalize_kernel<<<1, 1024, 0, st>>>(p.partials, blocks, p.B, losses);
  YNB_COUNT_LAUNCH();
  return cudaGetLastError();
}

// ---- torch.optim.SGD(momentum, weight_decay), one step over a flat parameter vector ------------
// train.py:167-171,230.  d = g + wd*p;  buf = first ? d : m*buf + d;  p -= lr*buf.
// Same operation order as torch (add with alpha = one fused multiply-add), so the update is
// bit-identical to the CPU optimiser.  16-byte accesses, 3 reads + 2 writes per element.
__global__ void __launch_bounds__(256) sgd_step_kernel(float* __restrict__ p, const float* __restrict__ g,
                                                       float* __restrict__ buf, long long n, float lr, float momentum,
                                                       float wd, int first, float grad_scale) {
  const long long n4 = n >> 2;
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long nth = (long long)gridDim.x * blockDim.x;
  auto upd = [&](float pv, float gv, float bv, float& pn, float& bn) {
    const float gs = grad_scale == 1.0f ? gv : __fmul_rn(gv, grad_scale);
    const float d = wd != 0.0f ? __fmaf_rn(pv, wd, gs) : gs;
    bn = first ? d : __fadd_rn(__fmul_rn(bv, momentum), d);
    pn = __fmaf_rn(bn, -lr, pv);
  };
  for (long long i = tid; i < n4; i += nth) {
    const float4 pv = reinterpret_cast<const float4*>(p)[i];
    const float4 gv = reinterpret_cast<const float4*>(g)[i];
    float4 bv = first ? make_float4(0.f, 0.f, 0.f, 0.f) : reinterpret_cast<const float4*>(buf)[i];
    float4 pn, bn;
    upd(pv.x, gv.x, bv.x, pn.x, bn.x); upd(pv.y, gv.y, bv.y, pn.y, bn.y);
    upd(pv.z, gv.z, bv.z, pn.z, bn.z); upd(pv.w, gv.w, bv.w, pn.w, bn.w);
    reinterpret_cast<float4*>(p)[i] = pn;
    reinterpret_cast<float4*>(buf)[i] = bn;
  }
  for (long long i = (n4 << 2) + tid; i < n; i += nth) {
    float pn, bn;
    upd(p[i], g[i], first ? 0.0f : buf[i], pn, bn);
    p[i] = pn; buf[i] = bn;
  }
}

inline cudaError_t launch_sgd_step(float* p, const float* g, float* buf, long long n, float lr, float momentum,
                                   float wd, int first, float grad_scale, cudaStream_t st) {
  long long need = ((n >> 2) + 255) / 256;
  if (need < 1) need = 1;
  const int blocks = (int)(need < kNumSMs * 8 ? need : kNumSMs * 8);
  sgd_step_kernel<<<blocks, 256, 0, st>>>(p, g, buf, n, lr, momentum, wd, first, grad_scale);
  YNB_COUNT_LAUNCH();
  return cudaGetLastError();
}

// ---- ModelEMA.update (utils/misc.py:78-86) over EVERY floating-point state tensor in ONE launch -------------
//   v *= d;  v += (1 - d) * m      per tensor in the reference: ~2 x 469 ATen launches per training step.
// Here: a device table of (ema pointer, model pointer, element count) and a chunk map; one CTA walks chunks of
// kEmaChunk elements.  Same two roundings as the reference's in-place ops (no FMA contraction; the Python scalars
// d and 1 - d reach the tensor op as float32), so the result is bit-identical.
constexpr int kEmaChunk = 2048;

__global__ void __launch_bounds__(256) ema_update_kernel(const unsigned long long* __restrict__ ema_ptrs,
                                                         const unsigned long long* __restrict__ model_ptrs,
                                                         const long long* __restrict__ sizes,
                                                         const int* __restrict__ chunk_tensor,
                                                         const int* __restrict__ chunk_index, int num_chunks, float d,
                                                         float one_minus_d) {
  for (int c = blockIdx.x; c < num_chunks; c += gridDim.x) {
    const int t = chunk_tensor[c];
    float* __restrict__ v = reinterpret_cast<float*>(ema_ptrs[t]);
    const float* __restrict__ m = reinterpret_cast<const float*>(model_ptrs[t]);
    const long long begin = (long long)chunk_index[c] * kEmaChunk;
    const long long end = min(begin + kEmaChunk, sizes[t]);
    const bool vec = ((ema_ptrs[t] | model_ptrs[t]) & 15ull) == 0;
    if (vec) {
      const long long n4 = (end - begin) >> 2;
      for (long long i = threadIdx.x; i < n4; i += blockDim.x) {
        float4 a = reinterpret_cast<float4*>(v + begin)[i];
        const float4 b = __ldg(reinterpret_cast<const float4*>(m + begin) + i);
        a.x = __fadd_rn(__fmul_rn(a.x, d), __fmul_rn(one_minus_d, b.x));
        a.y = __fadd_rn(__fmul_rn(a.y, d), __fmul_rn(one_minus_d, b.y));
        a.z = __fadd_rn(__fmul_rn(a.z, d), __fmul_rn(one_minus_d, b.z));
        a.w = __fadd_rn(__fmul_rn(a.w, d), __fmul_rn(one_minus_d, b.w));
        reinterpret_cast<float4*>(v + begin)[i] = a;
      }
      for (long long i = begin + (n4 << 2) + threadIdx.x; i < end; i += blockDim.x)
        v[i] = __fadd_rn(__fmul_rn(v[i], d), __fmul_rn(one_minus_d, __ldg(m + i)));
    } else {
      for (long long i = begin + threadIdx.x; i < end; i += blockDim.x)
        v[i] = __fadd_rn(__fmul_rn(v[i], d), __fmul_rn(one_minus_d, __ldg(m + i)));
    }
  }
}

inline cudaError_t launch_ema_update(const unsigned long long* ema_ptrs, const unsigned long long* model_ptrs,
                                     const long long* sizes, const int* chunk_tensor, const int* chunk_index,
                                     int num_chunks, float d, float one_minus_d, cudaStream_t st) {
  if (num_chunks <= 0) return cudaSuccess;
  const int blocks = num_chunks < kNumSMs * 8 ? num_chunks : kNumSMs * 8;
  ema_update_kernel<<<blocks, 256, 0, st>>>(ema_ptrs, model_ptrs, sizes, chunk_tensor, chunk_index, num_chunks, d,
                                            one_minus_d);
  YNB_COUNT_LAUNCH();
  return cudaGetLastError();
}

// ---- tools.multi_gt_creator (tools.py:97-216) on the device ----------------------------------------
// labels [B, L, 5] float32 = xmin, ymin, xmax, ymax (normalised), class; counts [B].
// One thread per image walks its labels IN ORDER (later labels overwrite earlier ones on the same
// cell / anchor, as the reference's Python loop does); float64 arithmetic in the reference's
// operation order (no FMA contraction), cast to float32 on store.  target must be zeroed before.
struct TargetParams {
  const float* labels;
  const int* counts;
  float* target;           // [B, N, 11]
  int B, L, A, S;
  int grid[3], stride[3];
  long long row_off[3];    // first anchor row of each level
  long long N;
  double anchors[3 * kTrainMaxAnchors][2];
};

__global__ void build_targets_kernel(const TargetParams p) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= p.B) return;
  const int n = p.counts ? min(p.counts[b], p.L) : p.L;
  const double w = (double)p.S, h = (double)p.S;
  const int na = 3 * p.A;
  float* __restrict__ tg = p.target + (long long)b * p.N * 11;
  for (int i = 0; i < n; ++i) {
    const float* lab = p.labels + ((long long)b * p.L + i) * 5;
    const double xmin = lab[0], ymin = lab[1], xmax = lab[2], ymax = lab[3];
    const int cls = (int)lab[4];
    const double cx = __dmul_rn(__dadd_rn(xmax, xmin) / 2.0, w), cy = __dmul_rn(__dadd_rn(ymax, ymin) / 2.0, h);
    const double bw = __dmul_rn(__dsub_rn(xmax, xmin), w), bh = __dmul_rn(__dsub_rn(ymax, ymin), h);
    if (bw < 1.0 || bh < 1.0) continue;                       // "dirty data" (:120-122)
    // compute_iou (tools.py:37-77) of [0,0,aw,ah] against [0,0,bw,bh]
    double best_iou = 0.0;
    int best = 0;
    unsigned above = 0;
    for (int k = 0; k < na; ++k) {
      const double aw = p.anchors[k][0], ah = p.anchors[k][1];
      const double iw = __dsub_rn(fmin(0.0 + bw / 2.0, 0.0 + aw / 2.0), fmax(0.0 - bw / 2.0, 0.0 - aw / 2.0));
      const double ih = __dsub_rn(fmin(0.0 + bh / 2.0, 0.0 + ah / 2.0), fmax(0.0 - bh / 2.0, 0.0 - ah / 2.0));
      const double si = __dmul_rn(ih, iw);
      const double u = __dadd_rn(__dsub_rn(__dadd_rn(__dmul_rn(bw, bh), __dmul_rn(aw, ah)), si), 1e-20);
      const double iou = si / u;
      if (k == 0 || iou > best_iou) { best_iou = iou; best = k; }      // np.argmax: first maximum
      if (iou > 0.5) above |= 1u << k;                                  // IGNORE_THRESH (data/config.py:3)
    }
    for (int k = 0; k < na; ++k) {
      if (!(k == best || ((above >> k) & 1u))) continue;
      const int lvl = k / p.A, a = k - lvl * p.A;
      const double s = (double)p.stride[lvl];
      const double cxs = cx / s, cys = cy / s;
      const int gx = (int)cxs, gy = (int)cys;
      if (gx >= p.grid[lvl] || gy >= p.grid[lvl]) continue;   // :147,:186 (the reference raises for ignored ones)
      float* t = tg + (p.row_off[lvl] + ((long long)gy * p.grid[lvl] + gx) * p.A + a) * 11;
      if (k == best) {
        t[0] = 1.0f;
        t[1] = (float)cls;
        t[2] = (float)__dsub_rn(cxs, (double)gx);
        t[3] = (float)__dsub_rn(cys, (double)gy);
        t[4] = (float)log(bw / p.anchors[k][0]);
        t[5] = (float)log(bh / p.anchors[k][1]);
        t[6] = (float)__dsub_rn(2.0, __dmul_rn(bw / w, bh / h));
        t[7] = (float)xmin; t[8] = (float)ymin; t[9] = (float)xmax; t[10] = (float)ymax;
      } else {
        t[0] = -1.0f;
        t[6] = -1.0f;
      }
    }
  }
}

inline cudaError_t launch_build_targets(const TargetParams& p, cudaStream_t st) {
  cudaError_t e = cudaMemsetAsync(p.target, 0, (size_t)p.B * p.N * 11 * sizeof(float), st);
  if (e != cudaSuccess) return e;
  build_targets_kernel<<<(p.B + 31) / 32, 32, 0, st>>>(p);
  YNB_COUNT_LAUNCH();
  return cudaGetLastError();
}

// ---- backward of the depthwise 3x3 convolution (config 5: "backward of the dw/pw conv kernels") -----
// Forward (ynb_dwconv3x3): out[b,y,x,c] = bias[c] + sum_t w[t][c] * in[b, y*s+dy-1, x*s+dx-1, c].
//   dIn[b,yi,xi,c] = sum_t w[t][c] * dOut[b, (yi+1-dy)/s, (xi+1-dx)/s, c]   (where divisible and inside)
// Stride 1 is the forward convolution of dOut with the taps reversed: it runs on the TMA halo-tile kernel
// of the forward path (dwconv3x3_tma_kernel<1, true>).  This kernel is the stride-2 / unaligned path:
// NHWC, a thread owns 4 channels of one input pixel (16-byte accesses when VEC).
template <bool VEC>
__global__ void __launch_bounds__(256) dwconv3x3_bwd_data_kernel(const float* __restrict__ dout, int do_ld, int do_off,
                                                                 float* __restrict__ din, int di_ld, int di_off,
                                                                 const float* __restrict__ w, int B, int h_in, int w_in,
                                                                 int C, int stride) {
  const int c4n = (C + 3) >> 2;
  const int h_out = (h_in - 1) / stride + 1, w_out = (w_in - 1) / stride + 1;
  const long long total = (long long)B * h_in * w_in * c4n;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c4 = (int)(i % c4n);
    long long pix = i / c4n;
    const int xi = (int)(pix % w_in);
    pix /= w_in;
    const int yi = (int)(pix % h_in);
    const int b = (int)(pix / h_in);
    const int c = c4 * 4;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int dy = 0; dy < 3; ++dy) {
      const int ty = yi + 1 - dy;
      if (ty < 0 || ty % stride) continue;
      const int yo = ty / stride;
      if (yo >= h_out) continue;
#pragma unroll
      for (int dx = 0; dx < 3; ++dx) {
        const int txx = xi + 1 - dx;
        if (txx < 0 || txx % stride) continue;
        const int xo = txx / stride;
        if (xo >= w_out) continue;
        const float* dp = dout + (((long long)b * h_out + yo) * w_out + xo) * do_ld + do_off + c;
        const float* wp = w + (dy * 3 + dx) * C + c;
        if (VEC) {
          const float4 d = *reinterpret_cast<const float4*>(dp);
          const float4 k = __ldg(reinterpret_cast<const float4*>(wp));
          acc[0] = fmaf(k.x, d.x, acc[0]); acc[1] = fmaf(k.y, d.y, acc[1]);
          acc[2] = fmaf(k.z, d.z, acc[2]); acc[3] = fmaf(k.w, d.w, acc[3]);
        } else {
#pragma unroll
          for (int k = 0; k < 4; ++k)
            if (c + k < C) acc[k] = fmaf(wp[k], dp[k], acc[k]);
        }
      }
    }
    float* op = din + (((long long)b * h_in + yi) * w_in + xi) * di_ld + di_off + c;
    if (VEC) {
      *reinterpret_cast<float4*>(op) = make_float4(acc[0], acc[1], acc[2], acc[3]);
    } else {
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (c + k < C) op[k] = acc[k];
    }
  }
}

// Stride 2, aligned views: a thread owns the 2 x 2 input block (2p..2p+1, 2q..2q+1) of 4 channels.  By
// parity an input pixel receives 1 / 2 / 2 / 4 taps, all from the four outputs (p..p+1, q..q+1): 4 loads
// and 9 FMAs per channel for 4 pixels (the generic kernel walks 9 guarded taps per pixel).  The 9 x C
// weights sit in shared memory.
__global__ void __launch_bounds__(256) dwconv3x3_s2_bwd_data_kernel(const float* __restrict__ dout, int do_ld, int do_off,
                                                                    float* __restrict__ din, int di_ld, int di_off,
                                                                    const float* __restrict__ w, int B, int h_in, int w_in,
                                                                    int C) {
  extern __shared__ __align__(16) float sw[];            // [9][C]
  for (int i = threadIdx.x; i < 9 * C; i += blockDim.x) sw[i] = w[i];
  __syncthreads();
  const int c4n = C >> 2;
  const int h_out = (h_in - 1) / 2 + 1, w_out = (w_in - 1) / 2 + 1;
  const int hb = (h_in + 1) >> 1, wb = (w_in + 1) >> 1;
  const long long total = (long long)B * hb * wb * c4n;
  const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % c4n) * 4;
    long long r = i / c4n;
    const int q = (int)(r % wb);
    r /= wb;
    const int pp = (int)(r % hb);
    const int b = (int)(r / hb);
    const float* d00p = dout + (((long long)b * h_out + pp) * w_out + q) * do_ld + do_off + c;
    const bool py = pp + 1 < h_out, qx = q + 1 < w_out;
    const float4 d00 = *reinterpret_cast<const float4*>(d00p);
    const float4 d01 = qx ? *reinterpret_cast<const float4*>(d00p + do_ld) : z4;
    const float4 d10 = py ? *reinterpret_cast<const float4*>(d00p + (long long)w_out * do_ld) : z4;
    const float4 d11 = (py && qx) ? *reinterpret_cast<const float4*>(d00p + (long long)(w_out + 1) * do_ld) : z4;
    float4 k[9];
#pragma unroll
    for (int t = 0; t < 9; ++t) k[t] = *reinterpret_cast<const float4*>(sw + t * C + c);
    auto mul = [](const float4& a, const float4& x) { return make_float4(a.x * x.x, a.y * x.y, a.z * x.z, a.w * x.w); };
    auto fma4 = [](const float4& a, const float4& x, const float4& y) {
      return make_float4(fmaf(a.x, x.x, y.x), fmaf(a.y, x.y, y.y), fmaf(a.z, x.z, y.z), fmaf(a.w, x.w, y.w));
    };
    // tap order = ascending (dy, dx) as in the generic kernel: identical rounding
    const float4 ee = mul(k[4], d00);
    const float4 eo = fma4(k[5], d00, mul(k[3], d01));
    const float4 oe = fma4(k[7], d00, mul(k[1], d10));
    const float4 oo = fma4(k[8], d00, fma4(k[6], d01, fma4(k[2], d10, mul(k[0], d11))));
    const int yi = 2 * pp, xi = 2 * q;
    float* o = din + (((long long)b * h_in + yi) * w_in + xi) * di_ld + di_off + c;
    const bool y1 = yi + 1 < h_in, x1 = xi + 1 < w_in;
    *reinterpret_cast<float4*>(o) = ee;
    if (x1) *reinterpret_cast<float4*>(o + di_ld) = eo;
    if (y1) *reinterpret_cast<float4*>(o + (long long)w_in * di_ld) = oe;
    if (y1 && x1) *reinterpret_cast<float4*>(o + (long long)(w_in + 1) * di_ld) = oo;
  }
}

//   dW[t][c] = sum_{b,y,x} dOut[b,y,x,c] * in[b, y*s+dy-1, x*s+dx-1, c];  dBias[c] = sum dOut[b,y,x,c]
// Work item = a segment of kDwSeg consecutive outputs of one output row.  A thread owns 4 channels
// (16-byte loads) and walks its segment with a 3x3 register window of the input that slides by
// `stride` columns (3 | 6 new loads per output instead of 9), accumulating its 10 float4 sums in
// registers over all the items of its slice; the block (16 channel groups x 8 slices) reduces the slices
// in shared memory and writes partial[blockIdx.x][10][C].  Stage 2 (reduce_partials_kernel) sums the
// blocks in fixed order: deterministic, no float atomics.
constexpr int kDwBwdCg = 16;       // 4-channel groups per block (64 channels)
constexpr int kDwBwdSlices = 8;
constexpr int kDwSeg = 16;
template <int STRIDE, bool VEC>
__global__ void __launch_bounds__(kDwBwdCg * kDwBwdSlices)
dwconv3x3_bwd_weight_kernel(const float* __restrict__ dout, int do_ld, int do_off, const float* __restrict__ in, int in_ld,
                            int in_off, float* __restrict__ partial, int B, int h_in, int w_in, int C) {
  const int h_out = (h_in - 1) / STRIDE + 1, w_out = (w_in - 1) / STRIDE + 1;
  const int segs = (w_out + kDwSeg - 1) / kDwSeg;
  const long long items = (long long)B * h_out * segs;
  const int c = (blockIdx.y * kDwBwdCg + threadIdx.x) * 4;
  float4 acc[10];
#pragma unroll
  for (int k = 0; k < 10; ++k) acc[k] = make_float4(0.f, 0.f, 0.f, 0.f);
  auto ld4 = [&](const float* q) -> float4 {
    if (VEC) return *reinterpret_cast<const float4*>(q);
    return make_float4(q[0], c + 1 < C ? q[1] : 0.f, c + 2 < C ? q[2] : 0.f, c + 3 < C ? q[3] : 0.f);
  };
  if (c < C) {
    for (long long it = (long long)blockIdx.x * kDwBwdSlices + threadIdx.y; it < items;
         it += (long long)gridDim.x * kDwBwdSlices) {
      const int seg = (int)(it % segs);
      const long long r = it / segs;
      const int b = (int)(r / h_out), yo = (int)(r % h_out);
      const int x0 = seg * kDwSeg, x1 = min(x0 + kDwSeg, w_out);
      const float* drow = dout + (((long long)b * h_out + yo) * w_out) * do_ld + do_off + c;
      const float* irow[3];
      bool rok[3];
#pragma unroll
      for (int dy = 0; dy < 3; ++dy) {
        const int yi = yo * STRIDE + dy - 1;
        rok[dy] = yi >= 0 && yi < h_in;
        irow[dy] = in + (((long long)b * h_in + (rok[dy] ? yi : 0)) * w_in) * in_ld + in_off + c;
      }
      float4 win[3][3];
      const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
      // columns x0*S-1, x0*S of the first window (the third arrives in the loop's load step)
#pragma unroll
      for (int dy = 0; dy < 3; ++dy) {
#pragma unroll
        for (int j = 0; j < 3 - STRIDE; ++j) {
          const int xi = x0 * STRIDE - 1 + j + (STRIDE - 1) * 0;
          win[dy][j + STRIDE] = (rok[dy] && xi >= 0 && xi < w_in) ? ld4(irow[dy] + (long long)xi * in_ld) : z4;
        }
      }
      for (int xo = x0; xo < x1; ++xo) {
#pragma unroll
        for (int dy = 0; dy < 3; ++dy) {
#pragma unroll
          for (int j = 0; j < 3 - STRIDE; ++j) win[dy][j] = win[dy][j + STRIDE];     // slide
#pragma unroll
          for (int j = 3 - STRIDE; j < 3; ++j) {
            const int xi = xo * STRIDE - 1 + j;
            win[dy][j] = (rok[dy] && xi >= 0 && xi < w_in) ? ld4(irow[dy] + (long long)xi * in_ld) : z4;
          }
        }
        const float4 d = ld4(drow + (long long)xo * do_ld);
        acc[9].x += d.x; acc[9].y += d.y; acc[9].z += d.z; acc[9].w += d.w;
#pragma unroll
        for (int dy = 0; dy < 3; ++dy)
#pragma unroll
          for (int dx = 0; dx < 3; ++dx) {
            float4& a = acc[dy * 3 + dx];
            const float4 v = win[dy][dx];
            a.x = fmaf(d.x, v.x, a.x); a.y = fmaf(d.y, v.y, a.y); a.z = fmaf(d.z, v.z, a.z); a.w = fmaf(d.w, v.w, a.w);
          }
      }
    }
  }
  __shared__ float4 sh[kDwBwdSlices][10][kDwBwdCg];
#pragma unroll
  for (int k = 0; k < 10; ++k) sh[threadIdx.y][k][threadIdx.x] = acc[k];
  __syncthreads();
  for (int k = threadIdx.y; k < 10; k += kDwBwdSlices) {
    float4 s4 = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int j = 0; j < kDwBwdSlices; ++j) {
      const float4 v = sh[j][k][threadIdx.x];
      s4.x += v.x; s4.y += v.y; s4.z += v.z; s4.w += v.w;
    }
    float* q = partial + ((long long)blockIdx.x * 10 + k) * C + c;
    const float vals[4] = {s4.x, s4.y, s4.z, s4.w};
#pragma unroll
    for (int e = 0; e < 4; ++e)
      if (c + e < C) q[e] = vals[e];
  }
}

// out[i] = sum_j partial[j][i]: 32 elements x 32 chunk slices per block, fixed summation order
// (deterministic second stage of the weight gradients; the slices keep the serial chain short).
constexpr int kRedSlices = 32;
__global__ void __launch_bounds__(32 * kRedSlices) reduce_partials_kernel(const float* __restrict__ partial, int chunks,
                                                                          long long elems, float* __restrict__ out) {
  __shared__ float sh[kRedSlices][33];
  const long long i = (long long)blockIdx.x * 32 + threadIdx.x;
  float s = 0.0f;
  if (i < elems)
    for (int j = threadIdx.y; j < chunks; j += kRedSlices) s += partial[(long long)j * elems + i];
  sh[threadIdx.y][threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.y == 0 && i < elems) {
    float t = 0.0f;
#pragma unroll
    for (int j = 0; j < kRedSlices; ++j) t += sh[j][threadIdx.x];
    out[i] = t;
  }
}
// Same for a partial made of two consecutive pieces per chunk (dW then db): ONE launch, two outputs.
__global__ void __launch_bounds__(32 * kRedSlices) reduce_partials2_kernel(const float* __restrict__ partial, int chunks,
                                                                           long long elems_a, float* __restrict__ out_a,
                                                                           long long elems_b, float* __restrict__ out_b) {
  __shared__ float sh[kRedSlices][33];
  const long long elems = elems_a + elems_b;
  const long long i = (long long)blockIdx.x * 32 + threadIdx.x;
  float s = 0.0f;
  if (i < elems)
    for (int j = threadIdx.y; j < chunks; j += kRedSlices) s += partial[(long long)j * elems + i];
  sh[threadIdx.y][threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.y == 0 && i < elems) {
    float t = 0.0f;
#pragma unroll
    for (int j = 0; j < kRedSlices; ++j) t += sh[j][threadIdx.x];
    if (i < elems_a) out_a[i] = t; else out_b[i - elems_a] = t;
  }
}
inline void launch_reduce_partials2(const float* partial, int chunks, long long ea, float* oa, long long eb, float* ob,
                                    cudaStream_t st) {
  reduce_partials2_kernel<<<(unsigned)((ea + eb + 31) / 32), dim3(32, kRedSlices), 0, st>>>(partial, chunks, ea, oa, eb, ob);
  YNB_COUNT_LAUNCH();
}
inline void launch_reduce_partials(const float* partial, int chunks, long long elems, float* out, cudaStream_t st) {
  reduce_partials_kernel<<<(unsigned)((elems + 31) / 32), dim3(32, kRedSlices), 0, st>>>(partial, chunks, elems, out);
  YNB_COUNT_LAUNCH();
}

inline int dw_bwd_chunks(int B, int h_out, int w_out) {
  const long long items = (long long)B * h_out * ((w_out + kDwSeg - 1) / kDwSeg);
  long long chunks = (items + kDwBwdSlices - 1) / kDwBwdSlices;
  if (chunks > kNumSMs * 3) chunks = kNumSMs * 3;
  return (int)(chunks < 1 ? 1 : chunks);
}

// ---- backward of the pointwise conv w.r.t. its weights -----------------------------------------------
// dW[n][k] = sum_m dOut[m, n] * in[m, k];  dBias[n] = sum_m dOut[m, n].   (dIn = dOut . W is the forward
// GEMM with the transposed weight matrix: ynb_pwconv / ynb_pwconv_tc.)
// A reduction over M (10^4 ... 10^6 pixels) into a small N x K matrix, fp32 FFMA: block = (chunk of M,
// 128 x 128 tile of (n, k)); 16-pixel slabs of dOut and in go through shared memory (next slab
// prefetched into registers while the current one is multiplied), each thread owns an 8 x 8 register
// tile (two 4-wide column groups 64 apart: conflict-free 16-byte shared loads).  partial[chunk][N][K] is
// summed in fixed order by reduce_partials_kernel.  This kernel serves the views that are not 16-byte aligned
// (aligned ones go to the cp.async variant below): scalar loads, through the read-only path (__ldg: 133 registers,
// plain loads 137, CUDA 12.9).
constexpr int kPwBwdTile = 128;
constexpr int kPwBwdSlab = 16;
__global__ void __launch_bounds__(256) pwconv_bwd_weight_kernel(const float* __restrict__ dout, int do_ld, int do_off,
                                                                const float* __restrict__ in, int in_ld, int in_off,
                                                                float* __restrict__ partial_w, float* __restrict__ partial_b,
                                                                long long M, int K, int N, long long m_per_chunk) {
  __shared__ __align__(16) float sd[kPwBwdSlab][kPwBwdTile];
  __shared__ __align__(16) float sx[kPwBwdSlab][kPwBwdTile];
  const int n0 = blockIdx.y * kPwBwdTile, k0 = blockIdx.z * kPwBwdTile;
  const long long m0 = (long long)blockIdx.x * m_per_chunk;
  const long long m1 = m0 + m_per_chunk < M ? m0 + m_per_chunk : M;
  const int tn = (threadIdx.x >> 4) * 4, tk = (threadIdx.x & 15) * 4;
  // loader role: 512 float4 per operand per slab = 2 per thread: row = idx / 32, col4 = idx % 32
  const int lr0 = threadIdx.x >> 5, lc = (threadIdx.x & 31) * 4;      // rows lr0 and lr0 + 8
  float2 acc[8][4];                                         // packed pairs along k: FFMA2 (2 fp32 FMAs per issue)
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = make_float2(0.0f, 0.0f);
  float bsum = 0.0f;                                        // threads 0..127 of k-tile 0: bias gradient
  float4 pd[2], px[2];
  auto fetch = [&](long long m) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const long long mm = m + lr0 + 8 * h;
      float4 d = make_float4(0.f, 0.f, 0.f, 0.f), x = d;
      if (mm < m1) {
        const float* dp = dout + mm * do_ld + do_off + n0 + lc;
        const float* xp = in + mm * in_ld + in_off + k0 + lc;
        if (n0 + lc < N) d.x = __ldg(dp);
        if (n0 + lc + 1 < N) d.y = __ldg(dp + 1);
        if (n0 + lc + 2 < N) d.z = __ldg(dp + 2);
        if (n0 + lc + 3 < N) d.w = __ldg(dp + 3);
        if (k0 + lc < K) x.x = __ldg(xp);
        if (k0 + lc + 1 < K) x.y = __ldg(xp + 1);
        if (k0 + lc + 2 < K) x.z = __ldg(xp + 2);
        if (k0 + lc + 3 < K) x.w = __ldg(xp + 3);
      }
      pd[h] = d; px[h] = x;
    }
  };
  fetch(m0);
  for (long long m = m0; m < m1; m += kPwBwdSlab) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      *reinterpret_cast<float4*>(&sd[lr0 + 8 * h][lc]) = pd[h];
      *reinterpret_cast<float4*>(&sx[lr0 + 8 * h][lc]) = px[h];
    }
    __syncthreads();
    if (m + kPwBwdSlab < m1) fetch(m + kPwBwdSlab);
#pragma unroll
    for (int r = 0; r < kPwBwdSlab; ++r) {
      const float4 d0 = *reinterpret_cast<const float4*>(&sd[r][tn]), d1 = *reinterpret_cast<const float4*>(&sd[r][tn + 64]);
      const float4 x0 = *reinterpret_cast<const float4*>(&sx[r][tk]), x1 = *reinterpret_cast<const float4*>(&sx[r][tk + 64]);
      const float dd[8] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
      const float2 xx[4] = {make_float2(x0.x, x0.y), make_float2(x0.z, x0.w), make_float2(x1.x, x1.y),
                            make_float2(x1.z, x1.w)};
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float2 d2 = make_float2(dd[i], dd[i]);
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = __ffma2_rn(d2, xx[j], acc[i][j]);
      }
    }
    if (blockIdx.z == 0 && threadIdx.x < kPwBwdTile) {
#pragma unroll
      for (int r = 0; r < kPwBwdSlab; ++r) bsum += sd[r][threadIdx.x];
    }
    __syncthreads();
  }
  float* pw = partial_w + (long long)blockIdx.x * N * K;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int n = n0 + tn + (i & 3) + (i >> 2) * 64;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int k = k0 + tk + (j & 3) + (j >> 2) * 64;
      const float2 a2 = acc[i][j >> 1];
      if (n < N && k < K) pw[(long long)n * K + k] = (j & 1) ? a2.y : a2.x;
    }
  }
  if (blockIdx.z == 0 && threadIdx.x < kPwBwdTile && n0 + threadIdx.x < N)
    partial_b[(long long)blockIdx.x * N + n0 + threadIdx.x] = bsum;
}

// Aligned views (the product layouts): the same tile computation fed by a 4-stage cp.async pipeline — the
// slabs go global -> shared without passing through registers, three slabs (48 pixels x 2 operands) are
// in flight per block while one is multiplied, which covers the DRAM latency that the register-prefetch
// variant above exposes (one slab of lookahead, 1 block per SM).  2 blocks per SM.
constexpr int kPwBwdStages = 4;
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc, int src_bytes) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(gsrc), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__global__ void __launch_bounds__(256, 2) pwconv_bwd_weight_async_kernel(const float* __restrict__ dout, int do_ld, int do_off,
                                                                         const float* __restrict__ in, int in_ld, int in_off,
                                                                         float* __restrict__ partial_w,
                                                                         float* __restrict__ partial_b, long long M, int K,
                                                                         int N, long long m_per_chunk) {
  extern __shared__ __align__(16) float smem_pw[];          // [stages][2][16][128]
  auto sd = [&](int st, int r) { return smem_pw + ((st * 2 + 0) * kPwBwdSlab + r) * kPwBwdTile; };
  auto sx = [&](int st, int r) { return smem_pw + ((st * 2 + 1) * kPwBwdSlab + r) * kPwBwdTile; };
  const int n0 = blockIdx.y * kPwBwdTile, k0 = blockIdx.z * kPwBwdTile;
  const long long m0 = (long long)blockIdx.x * m_per_chunk;
  const long long m1 = m0 + m_per_chunk < M ? m0 + m_per_chunk : M;
  const int tn = (threadIdx.x >> 4) * 4, tk = (threadIdx.x & 15) * 4;
  const int lr0 = threadIdx.x >> 5, lc = (threadIdx.x & 31) * 4;
  const int nslab = m1 > m0 ? (int)((m1 - m0 + kPwBwdSlab - 1) / kPwBwdSlab) : 0;
  const bool dcol = n0 + lc < N, xcol = k0 + lc < K;        // N, K multiples of 4 here
  auto issue = [&](int slab) {
    if (slab < nslab) {
      const int st = slab % kPwBwdStages;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int r = lr0 + 8 * h;
        const long long mm = m0 + (long long)slab * kPwBwdSlab + r;
        const bool rok = mm < m1;
        const long long ms = rok ? mm : m0;                  // a valid address even when nothing is read
        cp_async16(sd(st, r) + lc, dout + ms * do_ld + do_off + n0 + (dcol ? lc : 0), rok && dcol ? 16 : 0);
        cp_async16(sx(st, r) + lc, in + ms * in_ld + in_off + k0 + (xcol ? lc : 0), rok && xcol ? 16 : 0);
      }
    }
    cp_async_commit();
  };
  float2 acc[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = make_float2(0.0f, 0.0f);
  float bsum = 0.0f;
#pragma unroll
  for (int sl = 0; sl < kPwBwdStages - 1; ++sl) issue(sl);
  for (int slab = 0; slab < nslab; ++slab) {
    cp_async_wait<kPwBwdStages - 2>();                       // slab `slab` has landed (this thread's copies)
    __syncthreads();                                         // ... everyone's; and slab - 1 is fully consumed
    issue(slab + kPwBwdStages - 1);                          // refills the stage slab - 1 used
    const int st = slab % kPwBwdStages;
#pragma unroll
    for (int r = 0; r < kPwBwdSlab; ++r) {
      const float4 d0 = *reinterpret_cast<const float4*>(sd(st, r) + tn), d1 = *reinterpret_cast<const float4*>(sd(st, r) + tn + 64);
      const float4 x0 = *reinterpret_cast<const float4*>(sx(st, r) + tk), x1 = *reinterpret_cast<const float4*>(sx(st, r) + tk + 64);
      const float dd[8] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
      const float2 xx[4] = {make_float2(x0.x, x0.y), make_float2(x0.z, x0.w), make_float2(x1.x, x1.y),
                            make_float2(x1.z, x1.w)};
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float2 d2 = make_float2(dd[i], dd[i]);
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = __ffma2_rn(d2, xx[j], acc[i][j]);
      }
    }
    if (blockIdx.z == 0 && threadIdx.x < kPwBwdTile) {
#pragma unroll
      for (int r = 0; r < kPwBwdSlab; ++r) bsum += sd(st, r)[threadIdx.x];
    }
  }
  cp_async_wait<0>();
  float* pw = partial_w + (long long)blockIdx.x * N * K;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int n = n0 + tn + (i & 3) + (i >> 2) * 64;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int k = k0 + tk + (j & 3) + (j >> 2) * 64;
      const float2 a2 = acc[i][j >> 1];
      if (n < N && k < K) pw[(long long)n * K + k] = (j & 1) ? a2.y : a2.x;
    }
  }
  if (blockIdx.z == 0 && threadIdx.x < kPwBwdTile && n0 + threadIdx.x < N)
    partial_b[(long long)blockIdx.x * N + n0 + threadIdx.x] = bsum;
}
constexpr size_t kPwBwdAsyncSmem = (size_t)kPwBwdStages * 2 * kPwBwdSlab * kPwBwdTile * sizeof(float);   // 64 KB

inline int pw_bwd_chunks(long long M, int K, int N) {
  const int tiles = ((N + kPwBwdTile - 1) / kPwBwdTile) * ((K + kPwBwdTile - 1) / kPwBwdTile);
  long long chunks = (kNumSMs * 2 + tiles - 1) / tiles;       // 2 resident blocks per SM: one wave
  const long long max_chunks = (M + 4 * kPwBwdSlab - 1) / (4 * kPwBwdSlab);
  if (chunks > max_chunks) chunks = max_chunks;
  if (chunks < 1) chunks = 1;
  return (int)chunks;
}

// ---- BatchNorm2d in training mode (utils/modules.py:13, backbone/shufflenetv2.py:47-62; nn.BatchNorm2d
// defaults eps 1e-5, momentum 0.1) on NHWC views [M, ld], channels [off, off + C) -------------------------
// Forward: batch mean / biased variance per channel -> y = act((x - mean) * rstd * gamma + beta); running
// statistics updated with the UNBIASED variance as torch does.  Two streaming passes over x (statistics,
// apply) + a fixed-order second stage: deterministic.
// Column-sum kernel shared by forward statistics (a = x, b = x) and backward (a = dy_eff, b = x_hat):
//   partial[chunk][0][c] = sum_m a[m][c];  partial[chunk][1][c] = sum_m a[m][c] * b[m][c]
// MODE 0: a = x, b = x.   MODE 1: a = dy * act'(y), b = (x - mean) * rstd.
constexpr int kBnCg = 16, kBnSlices = 16;
template <int MODE>
__global__ void __launch_bounds__(kBnCg * kBnSlices)
bn_colsum_kernel(const float* __restrict__ x, int x_ld, int x_off, const float* __restrict__ dy, int dy_ld, int dy_off,
                 const float* __restrict__ y, int y_ld, int y_off, const float* __restrict__ mean,
                 const float* __restrict__ rstd, float slope, int use_act, float* __restrict__ partial, long long M, int C,
                 long long rows_per_chunk) {
  const int c = (blockIdx.y * kBnCg + threadIdx.x) * 4;
  const long long r0 = (long long)blockIdx.x * rows_per_chunk;
  const long long r1 = r0 + rows_per_chunk < M ? r0 + rows_per_chunk : M;
  float4 s1 = make_float4(0.f, 0.f, 0.f, 0.f), s2 = s1;
  if (c < C) {
    float4 mu = s1, rs = s1;
    if (MODE == 1) {
      mu = *reinterpret_cast<const float4*>(mean + c);
      rs = *reinterpret_cast<const float4*>(rstd + c);
    }
    for (long long m = r0 + threadIdx.y; m < r1; m += kBnSlices) {
      const float4 xv = *reinterpret_cast<const float4*>(x + m * x_ld + x_off + c);
      float4 a = xv, b = xv;
      if (MODE == 1) {
        a = *reinterpret_cast<const float4*>(dy + m * dy_ld + dy_off + c);
        if (use_act) {
          const float4 yv = *reinterpret_cast<const float4*>(y + m * y_ld + y_off + c);
          a.x *= yv.x > 0.f ? 1.f : slope; a.y *= yv.y > 0.f ? 1.f : slope;
          a.z *= yv.z > 0.f ? 1.f : slope; a.w *= yv.w > 0.f ? 1.f : slope;
        }
        b = make_float4((xv.x - mu.x) * rs.x, (xv.y - mu.y) * rs.y, (xv.z - mu.z) * rs.z, (xv.w - mu.w) * rs.w);
      }
      s1.x += a.x; s1.y += a.y; s1.z += a.z; s1.w += a.w;
      s2.x = fmaf(a.x, b.x, s2.x); s2.y = fmaf(a.y, b.y, s2.y); s2.z = fmaf(a.z, b.z, s2.z); s2.w = fmaf(a.w, b.w, s2.w);
    }
  }
  __shared__ float4 sh[kBnSlices][2][kBnCg];
  sh[threadIdx.y][0][threadIdx.x] = s1;
  sh[threadIdx.y][1][threadIdx.x] = s2;
  __syncthreads();
  if (threadIdx.y < 2 && c < C) {
    float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int j = 0; j < kBnSlices; ++j) {
      const float4 v = sh[j][threadIdx.y][threadIdx.x];
      t.x += v.x; t.y += v.y; t.z += v.z; t.w += v.w;
    }
    *reinterpret_cast<float4*>(partial + ((long long)blockIdx.x * 2 + threadIdx.y) * C + c) = t;
  }
}

// sums[2][C] (float) -> mean, rstd, running statistics; double for the E[x^2] - mean^2 cancellation.
__global__ void bn_finalize_kernel(const float* __restrict__ sums, long long M, int C, float eps, float momentum,
                                   float* __restrict__ save_mean, float* __restrict__ save_rstd,
                                   float* __restrict__ running_mean, float* __restrict__ running_var) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const double mean = (double)sums[c] / (double)M;
  double var = (double)sums[C + c] / (double)M - mean * mean;
  if (var < 0.0) var = 0.0;
  save_mean[c] = (float)mean;
  save_rstd[c] = (float)(1.0 / sqrt(var + (double)eps));
  if (running_mean) running_mean[c] = (1.0f - momentum) * running_mean[c] + momentum * (float)mean;
  if (running_var) {
    const double unbiased = M > 1 ? var * (double)M / (double)(M - 1) : var;
    running_var[c] = (1.0f - momentum) * running_var[c] + momentum * (float)unbiased;
  }
}

// reduce_partials + bn_finalize in ONE launch (forward): block = 32 channels x kRedSlices chunk slices, both sums of a
// channel reduced in the SAME order as reduce_partials_kernel (bit-identical statistics), then the finalize arithmetic.
__global__ void __launch_bounds__(32 * kRedSlices)
bn_reduce_finalize_kernel(const float* __restrict__ partial, int chunks, long long M, int C, float eps, float momentum,
                          float* __restrict__ sums, float* __restrict__ save_mean, float* __restrict__ save_rstd,
                          float* __restrict__ running_mean, float* __restrict__ running_var) {
  __shared__ float sh[2][kRedSlices][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  const long long elems = 2LL * C;
  float s0 = 0.0f, s1 = 0.0f;
  if (c < C)
    for (int j = threadIdx.y; j < chunks; j += kRedSlices) {
      s0 += partial[(long long)j * elems + c];
      s1 += partial[(long long)j * elems + C + c];
    }
  sh[0][threadIdx.y][threadIdx.x] = s0;
  sh[1][threadIdx.y][threadIdx.x] = s1;
  __syncthreads();
  if (threadIdx.y == 0 && c < C) {
    float t0 = 0.0f, t1 = 0.0f;
#pragma unroll
    for (int j = 0; j < kRedSlices; ++j) { t0 += sh[0][j][threadIdx.x]; t1 += sh[1][j][threadIdx.x]; }
    sums[c] = t0;
    sums[C + c] = t1;
    const double mean = (double)t0 / (double)M;
    double var = (double)t1 / (double)M - mean * mean;
    if (var < 0.0) var = 0.0;
    save_mean[c] = (float)mean;
    save_rstd[c] = (float)(1.0 / sqrt(var + (double)eps));
    if (running_mean) running_mean[c] = (1.0f - momentum) * running_mean[c] + momentum * (float)mean;
    if (running_var) {
      const double unbiased = M > 1 ? var * (double)M / (double)(M - 1) : var;
      running_var[c] = (1.0f - momentum) * running_var[c] + momentum * (float)unbiased;
    }
  }
}

// MODE 0: y = act((x - mean) * rstd * gamma + beta)
// MODE 1: dx = gamma * rstd * (dy_eff - sum(dy_eff) / M - x_hat * sum(dy_eff * x_hat) / M);  sums = [dbeta | dgamma]
template <int MODE>
__global__ void __launch_bounds__(256)
bn_apply_kernel(const float* __restrict__ x, int x_ld, int x_off, const float* __restrict__ dy, int dy_ld, int dy_off,
                const float* __restrict__ y, int y_ld, int y_off, float* __restrict__ out, int o_ld, int o_off,
                const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ mean,
                const float* __restrict__ rstd, const float* __restrict__ sums, float slope, int act, long long M, int C) {
  const int c4n = C >> 2;
  const long long total = M * c4n;
  const float invM = 1.0f / (float)M;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long m = i / c4n;
    const int c = (int)(i - m * c4n) * 4;
    const float4 xv = *reinterpret_cast<const float4*>(x + m * x_ld + x_off + c);
    const float4 mu = __ldg(reinterpret_cast<const float4*>(mean + c)), rs = __ldg(reinterpret_cast<const float4*>(rstd + c));
    const float4 ga = __ldg(reinterpret_cast<const float4*>(gamma + c));
    const float xs[4] = {xv.x, xv.y, xv.z, xv.w}, mus[4] = {mu.x, mu.y, mu.z, mu.w}, rss[4] = {rs.x, rs.y, rs.z, rs.w};
    const float gas[4] = {ga.x, ga.y, ga.z, ga.w};
    float o[4];
    if (MODE == 0) {
      const float4 be = __ldg(reinterpret_cast<const float4*>(beta + c));
      const float bes[4] = {be.x, be.y, be.z, be.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float v = (xs[k] - mus[k]) * rss[k] * gas[k] + bes[k];
        o[k] = act == YNB_ACT_NONE ? v : (v > 0.f ? v : slope * v);
      }
    } else {
      const float4 dv = *reinterpret_cast<const float4*>(dy + m * dy_ld + dy_off + c);
      float ds[4] = {dv.x, dv.y, dv.z, dv.w};
      if (act != YNB_ACT_NONE) {
        const float4 yv = *reinterpret_cast<const float4*>(y + m * y_ld + y_off + c);
        const float ys[4] = {yv.x, yv.y, yv.z, yv.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) ds[k] *= ys[k] > 0.f ? 1.f : slope;
      }
      const float4 sb = __ldg(reinterpret_cast<const float4*>(sums + c)), sg = __ldg(reinterpret_cast<const float4*>(sums + C + c));
      const float sbs[4] = {sb.x, sb.y, sb.z, sb.w}, sgs[4] = {sg.x, sg.y, sg.z, sg.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float xh = (xs[k] - mus[k]) * rss[k];
        o[k] = gas[k] * rss[k] * (ds[k] - sbs[k] * invM - xh * sgs[k] * invM);
      }
    }
    *reinterpret_cast<float4*>(out + m * o_ld + o_off + c) = make_float4(o[0], o[1], o[2], o[3]);
  }
}

inline int bn_chunks(long long M) {
  long long chunks = (M + kBnSlices * 4 - 1) / (kBnSlices * 4);
  if (chunks > kNumSMs * 4) chunks = kNumSMs * 4;
  return (int)(chunks < 1 ? 1 : chunks);
}

// dOut *= act'(out)  in place is avoided: writes dPre[m, c] = dOut[m, c] * (out > 0 ? 1 : slope), slope = 0
// (ReLU) or 0.1 (LeakyReLU), for channel ranges given as (ld, off).  `out` is the forward OUTPUT (its sign
// equals the sign of the pre-activation for both activations).
__global__ void __launch_bounds__(256) act_bwd_kernel(const float* __restrict__ dout, int do_ld, int do_off,
                                                      const float* __restrict__ out, int o_ld, int o_off,
                                                      float* __restrict__ dpre, int dp_ld, int dp_off, long long M, int C,
                                                      float slope) {
  const long long total = M * C;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long m = i / C;
    const int c = (int)(i - m * C);
    const float o = out[m * o_ld + o_off + c];
    dpre[m * dp_ld + dp_off + c] = dout[m * do_ld + do_off + c] * (o > 0.0f ? 1.0f : slope);
  }
}

}  // namespace ynb

// =====================================================================================================
// Round 2: the pieces the chained training step (config 5) still lacked as callable entries.
// =====================================================================================================
namespace ynb {

// ---- stem conv (backbone/shufflenetv2.py:109-113): Conv2d(3, 24, 3, stride 2, pad 1, bias=False), UNFUSED ---------
// Training needs the pre-BatchNorm conv output (batch statistics), so the fused stem_pool_kernel does not apply.
//   x NCHW [B,3,S,S];  w [27][24] (index (ci*9 + ky*3 + kx)*24 + co, as the inference stem);  out NHWC [B,S/2,S/2,24]
__global__ void __launch_bounds__(256)
stem_conv_fwd_kernel(const float* __restrict__ x, const float* __restrict__ w, float* __restrict__ out, int B, int S) {
  __shared__ float s_w[27 * 24];
  for (int i = threadIdx.x; i < 27 * 24; i += 256) s_w[i] = w[i];
  __syncthreads();
  const int Hc = S / 2;
  const long long total = (long long)B * Hc * Hc * 6;             // 4 channels per thread
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
    const int g = (int)(i % 6);
    const long long pix = i / 6;
    const int xo = (int)(pix % Hc), yo = (int)((pix / Hc) % Hc), b = (int)(pix / ((long long)Hc * Hc));
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int ci = 0; ci < 3; ++ci)
#pragma unroll
      for (int ky = 0; ky < 3; ++ky) {
        const int yi = 2 * yo + ky - 1;
        if (yi < 0 || yi >= S) continue;
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
          const int xi = 2 * xo + kx - 1;
          if (xi < 0 || xi >= S) continue;
          const float v = __ldg(x + (((size_t)b * 3 + ci) * S + yi) * S + xi);
          const float4 k = *reinterpret_cast<const float4*>(s_w + (ci * 9 + ky * 3 + kx) * 24 + 4 * g);
          acc.x = fmaf(v, k.x, acc.x); acc.y = fmaf(v, k.y, acc.y); acc.z = fmaf(v, k.z, acc.z); acc.w = fmaf(v, k.w, acc.w);
        }
      }
    *reinterpret_cast<float4*>(out + pix * 24 + 4 * g) = acc;
  }
}

// dW[tap][co] = sum over output pixels of dout[pix][co] * x[pix shifted by tap]  (27 x 24 outputs, ~10^6 pixels).
// Work item = a segment of <= 128 output pixels of one output row: the 9 input rows (3 channels x 3 filter rows) it
// touches and its d out rows are staged in shared memory with coalesced loads; thread = (half, tap, group of 4 output
// channels) of 2 x 27 x 6 = 324, one 4-byte and one 16-byte shared load per 4 FMAs; the two halves take alternate
// pixels.  A block walks its items in a fixed order; per-(block, half) partials, fixed-order second stage.
constexpr int kStemWgOut = 27 * 24;
constexpr int kStemWgTW = 128;
constexpr int kStemWgThreads = 352;
__global__ void __launch_bounds__(kStemWgThreads)
stem_conv_bwd_weight_kernel(const float* __restrict__ dout, const float* __restrict__ x, float* __restrict__ partial, int B,
                            int S, int items, int nseg) {
  __shared__ float in_s[9][2 * kStemWgTW + 2];
  __shared__ float4 dy_s[kStemWgTW][6];
  const int Hc = S / 2;
  const int t = threadIdx.x;
  const bool active = t < 324;
  const int h = t / 162, r = t - h * 162;
  const int tap = r / 6, cg = r - tap * 6;
  const int row_s = (tap / 9) * 3 + (tap % 9) / 3, kx = tap % 3;
  const float4* dout4 = reinterpret_cast<const float4*>(dout);
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int item = blockIdx.x; item < items; item += gridDim.x) {
    const int seg = item % nseg, row = item / nseg;
    const int yo = row % Hc, b = row / Hc;
    const int x0 = seg * kStemWgTW, tw = min(kStemWgTW, Hc - x0);
    const int ncols = 2 * tw + 1;
    __syncthreads();
    for (int i = t; i < 9 * ncols; i += kStemWgThreads) {
      const int rr = i / ncols, cc = i - rr * ncols;
      const int yi = 2 * yo + (rr % 3) - 1, xi = 2 * x0 - 1 + cc;
      float v = 0.f;
      if (yi >= 0 && yi < S && xi >= 0 && xi < S) v = __ldg(x + (((size_t)b * 3 + rr / 3) * S + yi) * S + xi);
      in_s[rr][cc] = v;
    }
    const size_t base4 = (((size_t)b * Hc + yo) * Hc + x0) * 6;
    for (int i = t; i < tw * 6; i += kStemWgThreads) (&dy_s[0][0])[i] = __ldg(dout4 + base4 + i);
    __syncthreads();
    if (active) {
#pragma unroll 4
      for (int p = h; p < tw; p += 2) {
        const float xv = in_s[row_s][2 * p + kx];
        const float4 d = dy_s[p][cg];
        acc.x = fmaf(xv, d.x, acc.x); acc.y = fmaf(xv, d.y, acc.y);
        acc.z = fmaf(xv, d.z, acc.z); acc.w = fmaf(xv, d.w, acc.w);
      }
    }
  }
  if (active)
    *reinterpret_cast<float4*>(partial + ((size_t)blockIdx.x * 2 + h) * kStemWgOut + tap * 24 + cg * 4) = acc;
}
inline int stem_wg_nseg(int S) { return (S / 2 + kStemWgTW - 1) / kStemWgTW; }
inline int stem_wg_grid(int B, int S) {
  const long long items = (long long)B * (S / 2) * stem_wg_nseg(S);
  return (int)std::min<long long>(items, (long long)kNumSMs * 4);
}
inline int stem_wg_chunks(int B, int S) { return 2 * stem_wg_grid(B, S); }     // partial rows of 648 floats

// ---- MaxPool2d(3, stride 2, pad 1) on NHWC (backbone/shufflenetv2.py:116), forward and backward ------------------
__global__ void __launch_bounds__(256)
maxpool3x3s2_fwd_kernel(const float* __restrict__ in, float* __restrict__ out, int B, int H, int W, int C) {
  const int Ho = (H - 1) / 2 + 1, Wo = (W - 1) / 2 + 1, G = C / 4;
  const long long total = (long long)B * Ho * Wo * G;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
    const int g = (int)(i % G);
    const long long pix = i / G;
    const int xo = (int)(pix % Wo), yo = (int)((pix / Wo) % Ho), b = (int)(pix / ((long long)Wo * Ho));
    float4 m = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
    for (int ky = 0; ky < 3; ++ky) {
      const int yi = 2 * yo + ky - 1;
      if (yi < 0 || yi >= H) continue;
      for (int kx = 0; kx < 3; ++kx) {
        const int xi = 2 * xo + kx - 1;
        if (xi < 0 || xi >= W) continue;
        const float4 v = *reinterpret_cast<const float4*>(in + (((size_t)b * H + yi) * W + xi) * C + 4 * g);
        m.x = fmaxf(m.x, v.x); m.y = fmaxf(m.y, v.y); m.z = fmaxf(m.z, v.z); m.w = fmaxf(m.w, v.w);
      }
    }
    *reinterpret_cast<float4*>(out + pix * C + 4 * g) = m;
  }
}
// Backward, deterministic (no atomics): one thread per INPUT element looks at the <= 4 windows that contain it and
// takes d_out of those whose FIRST maximum (row-major scan, as ATen's max_pool2d_with_indices) is this element.
__global__ void __launch_bounds__(256)
maxpool3x3s2_bwd_kernel(const float* __restrict__ dout, const float* __restrict__ in, float* __restrict__ din, int B, int H,
                        int W, int C) {
  const int Ho = (H - 1) / 2 + 1, Wo = (W - 1) / 2 + 1;
  const long long total = (long long)B * H * W * C;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
    const int c = (int)(i % C);
    const long long pix = i / C;
    const int xi = (int)(pix % W), yi = (int)((pix / W) % H), b = (int)(pix / ((long long)W * H));
    const float me = in[i];
    float g = 0.0f;
    // windows (yo, xo) with 2*yo - 1 <= yi <= 2*yo + 1
    for (int yo = max(0, yi / 2); yo <= min(Ho - 1, (yi + 1) / 2); ++yo)
      for (int xo = max(0, xi / 2); xo <= min(Wo - 1, (xi + 1) / 2); ++xo) {
        bool first = true;                                 // is (yi, xi) the first maximum of this window?
        for (int ky = 0; ky < 3 && first; ++ky) {
          const int y2 = 2 * yo + ky - 1;
          if (y2 < 0 || y2 >= H) continue;
          for (int kx = 0; kx < 3; ++kx) {
            const int x2 = 2 * xo + kx - 1;
            if (x2 < 0 || x2 >= W) continue;
            const float v = in[(((size_t)b * H + y2) * W + x2) * C + c];
            const bool before = y2 < yi || (y2 == yi && x2 < xi);
            if (v > me || (before && v == me)) { first = false; break; }
          }
        }
        if (first) g += dout[(((size_t)b * Ho + yo) * Wo + xo) * C + c];
      }
    din[i] = g;
  }
}

// The same pair with the arg-max kept (what ATen's max_pool2d_with_indices does): forward also writes, per output
// element, which of the 9 taps (ky * 3 + kx, first maximum in row-major order) won; backward is then a gather — one
// thread per 4 input channels reads the <= 4 windows that contain its pixel (4 index bytes + 16 bytes of d out each).
__global__ void __launch_bounds__(256)
maxpool3x3s2_fwd_idx_kernel(const float* __restrict__ in, float* __restrict__ out, uint8_t* __restrict__ idx, int B, int H,
                            int W, int C) {
  const int Ho = (H - 1) / 2 + 1, Wo = (W - 1) / 2 + 1, G = C / 4;
  const long long total = (long long)B * Ho * Wo * G;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
    const int g = (int)(i % G);
    const long long pix = i / G;
    const int xo = (int)(pix % Wo), yo = (int)((pix / Wo) % Ho), b = (int)(pix / ((long long)Wo * Ho));
    float4 m = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
    uchar4 w = make_uchar4(255, 255, 255, 255);
    for (int ky = 0; ky < 3; ++ky) {
      const int yi = 2 * yo + ky - 1;
      if (yi < 0 || yi >= H) continue;
      for (int kx = 0; kx < 3; ++kx) {
        const int xi = 2 * xo + kx - 1;
        if (xi < 0 || xi >= W) continue;
        const float4 v = *reinterpret_cast<const float4*>(in + (((size_t)b * H + yi) * W + xi) * C + 4 * g);
        const unsigned char tp = (unsigned char)(ky * 3 + kx);
        if (v.x > m.x || w.x == 255) { m.x = v.x; w.x = tp; }
        if (v.y > m.y || w.y == 255) { m.y = v.y; w.y = tp; }
        if (v.z > m.z || w.z == 255) { m.z = v.z; w.z = tp; }
        if (v.w > m.w || w.w == 255) { m.w = v.w; w.w = tp; }
      }
    }
    *reinterpret_cast<float4*>(out + pix * C + 4 * g) = m;
    *reinterpret_cast<uchar4*>(idx + pix * C + 4 * g) = w;
  }
}
__global__ void __launch_bounds__(256)
maxpool3x3s2_bwd_idx_kernel(const float* __restrict__ dout, const uint8_t* __restrict__ idx, float* __restrict__ din, int B,
                            int H, int W, int C) {
  const int Ho = (H - 1) / 2 + 1, Wo = (W - 1) / 2 + 1, G = C / 4;
  const long long total = (long long)B * H * W * G;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
    const int g = (int)(i % G);
    const long long pix = i / G;
    const int xi = (int)(pix % W), yi = (int)((pix / W) % H), b = (int)(pix / ((long long)W * H));
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int yo = max(0, yi / 2); yo <= min(Ho - 1, (yi + 1) / 2); ++yo)          // ascending (yo, xo): fixed order
      for (int xo = max(0, xi / 2); xo <= min(Wo - 1, (xi + 1) / 2); ++xo) {
        const unsigned char me = (unsigned char)((yi - 2 * yo + 1) * 3 + (xi - 2 * xo + 1));
        const size_t o = (((size_t)b * Ho + yo) * Wo + xo) * C + 4 * g;
        const uchar4 w = *reinterpret_cast<const uchar4*>(idx + o);
        const float4 d = *reinterpret_cast<const float4*>(dout + o);
        if (w.x == me) s.x += d.x;
        if (w.y == me) s.y += d.y;
        if (w.z == me) s.z += d.z;
        if (w.w == me) s.w += d.w;
      }
    *reinterpret_cast<float4*>(din + pix * C + 4 * g) = s;
  }
}

// ---- ShuffleV2 unit data movement in the training step (backbone/shufflenetv2.py:14-28, 66-78) ---------------------
// x.chunk(2) with each half zero-padded from h to hp channels (forward) / its adjoint, and torch.cat + channel_shuffle
// (out[2i] = a[i], out[2i+1] = b[i]) / its adjoint: plain copies, one launch each instead of 4-6 ATen launches.
// op 0: split   x [M, 2h]            -> a, b [M, hp]   (a = x[:, :h], b = x[:, h:], zero pad)
// op 1: merge   a, b [M, hp]         -> x [M, 2h]      (adjoint of split: x[:, :h] = a[:, :h], x[:, h:] = b[:, :h])
// op 2: shuffle a, b [M, hp]         -> x [M, 2h]      (x[:, 2i] = a[:, i], x[:, 2i+1] = b[:, i])
// op 3: unshuffle x [M, 2h]          -> a, b [M, hp]   (adjoint of shuffle, zero pad)
__global__ void __launch_bounds__(256)
shuffle_unit_move_kernel(float* __restrict__ x, float* __restrict__ a, float* __restrict__ b, long long M, int h, int hp,
                         int op) {
  const long long total = M * hp;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
    const long long m = i / hp;
    const int c = (int)(i - m * hp);
    float* xr = x + m * 2 * h;
    if (op == 0) {
      a[i] = c < h ? xr[c] : 0.0f;
      b[i] = c < h ? xr[h + c] : 0.0f;
    } else if (op == 1) {
      if (c < h) { xr[c] = a[i]; xr[h + c] = b[i]; }
    } else if (op == 2) {
      if (c < h) *reinterpret_cast<float2*>(xr + 2 * c) = make_float2(a[i], b[i]);
    } else {
      float2 v = make_float2(0.0f, 0.0f);
      if (c < h) v = *reinterpret_cast<const float2*>(xr + 2 * c);
      a[i] = v.x;
      b[i] = v.y;
    }
  }
}

// ---- FPN / PAN merge backward (models/yolo_nano.py:291-296): out = a + resample(a2) => d a = d out (identity) and
//   mode 1 (a2 up-sampled x2, nearest):  d a2[y, x] = sum of the 2x2 block of d out
//   mode 2 (a2 down-sampled [::2, ::2]):  d a2[2y, 2x] = d out[y, x], zero elsewhere
// da2 has the shape of a2: (H/2 x W/2) in mode 1, (2H x 2W) in mode 2; H, W = the size of out.
__global__ void __launch_bounds__(256)
resample_bwd_kernel(const float* __restrict__ dout, float* __restrict__ da2, int B, int H, int W, int C, int mode) {
  const int H2 = mode == 1 ? H >> 1 : H << 1, W2 = mode == 1 ? W >> 1 : W << 1, G = C / 4;
  const long long total = (long long)B * H2 * W2 * G;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
    const int g = (int)(i % G);
    const long long pix = i / G;
    const int x = (int)(pix % W2), y = (int)((pix / W2) % H2), b = (int)(pix / ((long long)W2 * H2));
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    if (mode == 1) {
      for (int dy = 0; dy < 2; ++dy)
        for (int dx = 0; dx < 2; ++dx) {
          const int yy = 2 * y + dy, xx = 2 * x + dx;
          if (yy < H && xx < W) {
            const float4 v = *reinterpret_cast<const float4*>(dout + (((size_t)b * H + yy) * W + xx) * C + 4 * g);
            s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
          }
        }
    } else if (!(y & 1) && !(x & 1) && (y >> 1) < H && (x >> 1) < W) {
      s = *reinterpret_cast<const float4*>(dout + (((size_t)b * H + (y >> 1)) * W + (x >> 1)) * C + 4 * g);
    }
    *reinterpret_cast<float4*>(da2 + pix * C + 4 * g) = s;
  }
}

// out = a + b (gradient accumulation where a tensor feeds two consumers), 16 bytes per thread
__global__ void __launch_bounds__(256) add_kernel(const float* __restrict__ a, const float* __restrict__ b,
                                                   float* __restrict__ out, long long n4) {
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n4; i += (long long)gridDim.x * 256) {
    const float4 u = reinterpret_cast<const float4*>(a)[i], v = reinterpret_cast<const float4*>(b)[i];
    reinterpret_cast<float4*>(out)[i] = make_float4(u.x + v.x, u.y + v.y, u.z + v.z, u.w + v.w);
  }
}

inline unsigned grid_for(long long items) {
  long long blocks = (items + 255) / 256;
  if (blocks > (long long)kNumSMs * 16) blocks = (long long)kNumSMs * 16;
  return (unsigned)(blocks < 1 ? 1 : blocks);
}

}  // namespace ynb
