// COCO bbox AP on the device: the reference evaluator's results JSON (evaluator/cocoapi_evaluator.py) and
// pycocotools' COCOeval(cocoGt, cocoDt, 'bbox') evaluate + accumulate, with COCOeval's bbox defaults
// (T = 10 IoU thresholds, R = 101 recall thresholds, A = 4 area ranges, M = maxDets {1, 10, 100}).
//
//   append      engine rows after map_boxes -> one int32 row per results entry, in file order (image, kept row):
//               [image, class, score bits, x1, y1, x2, y2 bits].  The float32 values themselves: the JSON round trip
//               of Python floats is exact, so no decimal rounding is involved.
//   evaluate    1. cell order: stable LSD radix passes by score (descending), then by cell = (image rank, category
//                  index); a detection's position in its cell cuts the cell at maxDets[-1] = 100;
//               2. one block per cell: the bbIou matrix, then 40 independent greedy passes (4 ranges x 10
//                  thresholds) of evaluateImg -> per-detection TP / ignore bits; npig per (category, range);
//               3. per-category order: stable passes by score, then category, over the cell order (accumulate's
//                  concatenation in ascending image id followed by its mergesort);
//               4. one block per (category, range, maxDet, threshold): tp / fp scan, the precision envelope and the
//                  101 recall lookups -> precision [T,R,K,A,M], recall [T,K,A,M].
// Every float64 expression is written with explicit _rn intrinsics (the build contracts a*b+c into FMA otherwise),
// so precision and recall are bit-identical to pycocotools' float64 arithmetic.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <utility>

#include "common.cuh"
#include "voc_eval.cuh"

namespace ynb {
namespace coco {

constexpr int kRowInts = 7;
constexpr int kT = 10, kR = 101, kA = 4, kM = 3, kPairs = kT * kA;
constexpr int kMaxDet = 100;                 // maxDets[-1]: computeIoU / evaluateImg cut each cell here
constexpr int kPosShift = 40;                // m0 = TP bits [0, 40) | position in cell << 40

struct Thresholds {
  double iou[kT];                            // np.linspace(.5, .95, 10)
  double rec[kR];                            // np.linspace(0, 1, 101)
};

// areaRng = [[0, 1e10], [0, 32^2], [32^2, 96^2], [96^2, 1e10]], bounds inclusive.
__device__ __forceinline__ double area_lo(int a) { return a == 2 ? 1024.0 : a == 3 ? 9216.0 : 0.0; }
__device__ __forceinline__ double area_hi(int a) { return a == 1 ? 1024.0 : a == 2 ? 9216.0 : 1e10; }
__device__ __forceinline__ int max_det(int m) { return m == 0 ? 1 : m == 1 ? 10 : 100; }

__device__ __forceinline__ bool finite_bits(int32_t b) { return (((uint32_t)b >> 23) & 0xffu) != 0xffu; }

// Ascending order of the key is descending score; -0.0 and +0.0 share a key (equal scores keep input order).
__device__ __forceinline__ uint32_t score_desc_key(int32_t bits) {
  uint32_t u = (uint32_t)bits;
  if ((u & 0x7fffffffu) == 0) u = 0;
  const uint32_t asc = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
  return ~asc;
}

// ---- append -------------------------------------------------------------------------------------------------------
// One block per image: its first slot is state[0] + sum(counts[0..b)), as voc_append_kernel.
__global__ void __launch_bounds__(256)
coco_append_kernel(const float* __restrict__ boxes, const float* __restrict__ scores, const int* __restrict__ cls,
                   const int* __restrict__ counts, long long n_per_image, int image_base, int num_classes,
                   int* __restrict__ rows, long long capacity, long long* __restrict__ state) {
  __shared__ long long sm[8];
  const int b = blockIdx.x;
  long long before = 0;
  for (int i = threadIdx.x; i < b; i += blockDim.x) before += min((long long)max(counts[i], 0), n_per_image);
  long long tot;
  voc::block_exclusive_scan<long long, voc::AddOp, 256>(before, 0ll, voc::AddOp(), sm, &tot);
  const long long base = state[0] + tot;
  const long long cnt = min((long long)max(counts[b], 0), n_per_image);
  int bad = 0;
  for (long long k = threadIdx.x; k < cnt; k += blockDim.x) {
    const size_t src = (size_t)b * n_per_image + k;
    int row[kRowInts];
    row[0] = image_base + b;
    const int c = cls[src];
    bool ok = c >= 0 && c < num_classes;
    row[1] = ok ? c : 0;
    row[2] = __float_as_int(scores[src]);
    ok = finite_bits(row[2]) && ok;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      row[3 + j] = __float_as_int(boxes[src * 4 + j]);
      ok = finite_bits(row[3 + j]) && ok;
    }
    bad += !ok;
    const long long slot = base + k;
    if (slot < capacity) {
      int* dst = rows + (size_t)slot * kRowInts;
#pragma unroll
      for (int j = 0; j < kRowInts; ++j) dst[j] = row[j];
    }
  }
  if (bad) atomicAdd(reinterpret_cast<unsigned long long*>(state + 1), (unsigned long long)bad);
}

inline cudaError_t launch_coco_append(const float* boxes, const float* scores, const int* cls, const int* counts,
                                      int batch, long long n_per_image, int image_base, int num_classes, int* rows,
                                      long long capacity, long long* state, cudaStream_t st) {
  coco_append_kernel<<<batch, 256, 0, st>>>(boxes, scores, cls, counts, n_per_image, image_base, num_classes, rows,
                                            capacity, state);
  YNB_COUNT_LAUNCH();
  voc::voc_append_total_kernel<<<1, 256, 0, st>>>(counts, batch, n_per_image, state);
  YNB_COUNT_LAUNCH();
  return cudaGetLastError();
}

// ---- sort keys ----------------------------------------------------------------------------------------------------
// keys = score key of rows[src[i]] (src == nullptr: row i), vals = i.
__global__ void coco_score_keys_kernel(const int* __restrict__ rows, const uint32_t* __restrict__ src, long long n,
                                       uint32_t* __restrict__ keys, uint32_t* __restrict__ vals) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const long long r = src ? (long long)src[i] : i;
  keys[i] = score_desc_key(rows[(size_t)r * kRowInts + 2]);
  vals[i] = (uint32_t)i;
}

// keys = cell of the arena row vals[i]: image_rank * K + category index, or `cells` for a class without a category.
__global__ void coco_cell_keys_kernel(const int* __restrict__ rows, const uint32_t* __restrict__ vals, long long n,
                                      const int* __restrict__ image_rank, int num_images,
                                      const int* __restrict__ class_cat, int num_classes, int K,
                                      uint32_t* __restrict__ keys) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int* r = rows + (size_t)vals[i] * kRowInts;
  const int img = min(max(r[0], 0), num_images - 1), c = min(max(r[1], 0), num_classes - 1);
  const int k = class_cat[c];
  const long long cells = (long long)num_images * K;
  keys[i] = (uint32_t)(k < 0 ? cells : (long long)image_rank[img] * K + k);
}

// Cell ranges [cell_begin, cell_end) of the cell order (zeroed before: empty cells).
__global__ void coco_cell_bounds_kernel(const uint32_t* __restrict__ keys, long long n, long long cells,
                                        int* __restrict__ cell_begin, int* __restrict__ cell_end) {
  const long long d = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= n) return;
  const uint32_t c = keys[d];
  if (c >= cells) return;
  if (d == 0 || keys[d - 1] != c) cell_begin[c] = (int)d;
  if (d == n - 1 || keys[d + 1] != c) cell_end[c] = (int)d + 1;
}

// ---- evaluateImg --------------------------------------------------------------------------------------------------
// One block per cell (image rank, category).  Detections are the first <= 100 of the cell order (computeIoU's cut);
// GT are the cell's annotations in file order.  In range a, GT g is ignored when crowd or its area lies outside
// [lo, hi]; evaluateImg scans the GT with the non-ignored ones first, so its greedy choice for detection d at
// threshold t is: among GT not yet matched at (t, a) (crowd GT stay available) with IoU >= min(t, 1 - 1e-10), the
// largest IoU among non-ignored GT, later annotation on equal IoU; only if there is none, the same among ignored GT.
// A match on an ignored GT ignores d; an unmatched d is ignored when its own area lies outside the range.
constexpr int kMatchNT = 256;

__device__ __forceinline__ void warp_best(double& v, int& g) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double ov = __shfl_xor_sync(0xffffffffu, v, o);
    const int og = __shfl_xor_sync(0xffffffffu, g, o);
    if (ov > v || (ov == v && og > g)) { v = ov; g = og; }
  }
}

__global__ void __launch_bounds__(kMatchNT)
coco_match_kernel(const int* __restrict__ rows, const uint32_t* __restrict__ corder,
                  const int* __restrict__ cell_begin, const int* __restrict__ cell_end, int K,
                  const double* __restrict__ gt_boxes, const double* __restrict__ gt_area,
                  const uint8_t* __restrict__ gt_crowd, const int* __restrict__ gt_start, long long n_gt,
                  Thresholds thr, double* __restrict__ iou_ws, uint8_t* gtm, unsigned long long* __restrict__ m0,
                  unsigned long long* __restrict__ m1, int* __restrict__ npig) {
  __shared__ double dx[kMaxDet], dy[kMaxDet], dw[kMaxDet], dh[kMaxDet], da[kMaxDet];
  __shared__ unsigned long long tpm[kMaxDet], igm[kMaxDet];
  __shared__ int cnt[kA];
  const long long c = blockIdx.x;
  const int k = (int)(c % K), tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int gs = gt_start[c], G = gt_start[c + 1] - gs;
  const int ds = cell_begin[c], D = min(cell_end[c] - ds, kMaxDet);
  if (G == 0 && D <= 0) return;
  if (tid < kA) cnt[tid] = 0;
  __syncthreads();
  int mine[kA] = {0, 0, 0, 0};
  for (int g = tid; g < G; g += kMatchNT) {
    const double ar = gt_area[gs + g];
    const bool crowd = gt_crowd[gs + g];
#pragma unroll
    for (int a = 0; a < kA; ++a) mine[a] += !(crowd || ar < area_lo(a) || ar > area_hi(a));
  }
#pragma unroll
  for (int a = 0; a < kA; ++a)
    if (mine[a]) atomicAdd(&cnt[a], mine[a]);
  __syncthreads();
  if (tid < kA && cnt[tid]) atomicAdd(npig + k * kA + tid, cnt[tid]);
  if (D <= 0) return;
  for (int i = tid; i < D; i += kMatchNT) {
    const int* r = rows + (size_t)corder[ds + i] * kRowInts;
    const double x1 = (double)__int_as_float(r[3]), y1 = (double)__int_as_float(r[4]);
    const double x2 = (double)__int_as_float(r[5]), y2 = (double)__int_as_float(r[6]);
    dx[i] = x1;
    dy[i] = y1;
    dw[i] = __dsub_rn(x2, x1);                                // bbox = [x1, y1, x2 - x1, y2 - y1] in Python floats
    dh[i] = __dsub_rn(y2, y1);
    da[i] = __dmul_rn(dw[i], dh[i]);                          // loadRes: area = w * h
    tpm[i] = 0;
    igm[i] = 0;
  }
  __syncthreads();
  // maskUtils.iou (bbIou) into [D][G] at 100 * gs: each cell owns 100 rows of its GT's columns
  double* iou = iou_ws + (size_t)kMaxDet * gs;
  for (int e = tid; e < D * G; e += kMatchNT) {
    const int i = e / G, g = e - i * G;
    const double* gb = gt_boxes + (size_t)(gs + g) * 4;
    const double gx = gb[0], gy = gb[1], gw = gb[2], gh = gb[3];
    double v = 0.0;
    const double w = __dsub_rn(fmin(__dadd_rn(dw[i], dx[i]), __dadd_rn(gw, gx)), fmax(dx[i], gx));
    if (w > 0.0) {
      const double h = __dsub_rn(fmin(__dadd_rn(dh[i], dy[i]), __dadd_rn(gh, gy)), fmax(dy[i], gy));
      if (h > 0.0) {
        const double in = __dmul_rn(w, h);
        const double u = gt_crowd[gs + g] ? da[i] : __dsub_rn(__dadd_rn(da[i], __dmul_rn(gw, gh)), in);
        v = __ddiv_rn(in, u);
      }
    }
    iou[e] = v;
  }
  __syncthreads();
  for (int pair = warp; pair < kPairs; pair += kMatchNT / 32) {
    const int t = pair % kT, a = pair / kT;
    const double lo = area_lo(a), hi = area_hi(a), t_eff = fmin(thr.iou[t], 1.0 - 1e-10);
    const unsigned long long bit = 1ull << pair;
    uint8_t* matched = gtm + (size_t)pair * n_gt + gs;        // gtm[t, g] > 0 of (t, a)
    for (int i = 0; i < D; ++i) {
      double v1 = -1.0, v2 = -1.0;
      int g1 = -1, g2 = -1;
      for (int g = lane; g < G; g += 32) {
        const bool crowd = gt_crowd[gs + g];
        if (!crowd && matched[g]) continue;
        const double v = iou[(size_t)i * G + g];
        if (v < t_eff) continue;
        const double ar = gt_area[gs + g];
        if (crowd || ar < lo || ar > hi) {
          if (v >= v2) { v2 = v; g2 = g; }
        } else if (v >= v1) {
          v1 = v;
          g1 = g;
        }
      }
      warp_best(v1, g1);
      warp_best(v2, g2);
      if (lane == 0) {
        const int m = g1 >= 0 ? g1 : g2;
        if (m >= 0 && !gt_crowd[gs + m]) matched[m] = 1;
        if (g1 >= 0) atomicOr(&tpm[i], bit);
        else if (g2 >= 0 || da[i] < lo || da[i] > hi) atomicOr(&igm[i], bit);
      }
      __syncwarp();
    }
  }
  __syncthreads();
  for (int i = tid; i < D; i += kMatchNT) {
    m0[ds + i] = tpm[i] | ((unsigned long long)i << kPosShift);
    m1[ds + i] = igm[i];
  }
}

// ---- per-category order -------------------------------------------------------------------------------------------
// vals[i] = cell-order position q; keys = category index of q when q is kept (position < 100), else K (sorted last).
__global__ void coco_cat_keys_kernel(const uint32_t* __restrict__ ckey, const int* __restrict__ cell_begin,
                                     const uint32_t* __restrict__ vals, long long n, long long cells, int K,
                                     uint32_t* __restrict__ keys) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t q = vals[i], c = ckey[q];
  keys[i] = (c < cells && (long long)q - cell_begin[c] < kMaxDet) ? c % (uint32_t)K : (uint32_t)K;
}

// Category ranges [cstart, cend) and the gathered bits of each sorted position.
__global__ void coco_cat_gather_kernel(const uint32_t* __restrict__ keys, const uint32_t* __restrict__ vals,
                                       long long n, int K, const unsigned long long* __restrict__ m0,
                                       const unsigned long long* __restrict__ m1, unsigned long long* __restrict__ g0,
                                       unsigned long long* __restrict__ g1, int* __restrict__ cstart,
                                       int* __restrict__ cend) {
  const long long d = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= n) return;
  const uint32_t k = keys[d];
  if (k >= (uint32_t)K) return;
  g0[d] = m0[vals[d]];
  g1[d] = m1[vals[d]];
  if (d == 0 || keys[d - 1] != k) cstart[k] = (int)d;
  if (d == n - 1 || keys[d + 1] != k) cend[k] = (int)d + 1;
}

// ---- accumulate ---------------------------------------------------------------------------------------------------
// One block per (category k, range a, maxDet m, threshold t) walks the category's range from the END in chunks, as
// voc_class_ap_kernel: with the totals known, the cumsums at d are total - (count after d) and the envelope
// max(pr[d..]) is a forward max-scan in that walk order.  The sequence is the detections with position < maxDet;
// ignored ones keep their place and count in neither sum.
//   rc[d] = tp / npig,  pr[d] = tp / ((fp + tp) + 2^-52)
//   q[r]  = envelope at searchsorted(rc, recThrs[r], 'left'), 0 past the end: for recThrs[r] > 0 that index is the TP
//           d with rc[d-1] < recThrs[r] <= rc[d]; for recThrs[r] <= 0 it is the first d, whose envelope is max(pr).
//   recall = rc[-1] (tp total / npig, 0 without detections); both -1 when npig == 0.
__global__ void __launch_bounds__(voc::kApNT)
coco_accumulate_kernel(const unsigned long long* __restrict__ g0, const unsigned long long* __restrict__ g1,
                       const int* __restrict__ cstart, const int* __restrict__ cend, const int* __restrict__ npig_arr,
                       int K, Thresholds thr, double* __restrict__ precision, double* __restrict__ recall) {
  constexpr int NT = voc::kApNT, IT = voc::kApIT, CH = voc::kApChunk;
  __shared__ unsigned long long smc[NT / 32];
  __shared__ double smd[NT / 32];
  __shared__ double q[kR];
  const int b = blockIdx.x, tid = threadIdx.x;
  const int t = b % kT, m = (b / kT) % kM, a = (b / (kT * kM)) % kA, k = b / (kT * kM * kA);
  const int pair = a * kT + t, maxdet = max_det(m);
  const size_t rec_at = ((size_t)t * K + k) * (kA * kM) + a * kM + m;
  auto prec_at = [&](int r) { return (((size_t)t * kR + r) * K + k) * (kA * kM) + a * kM + m; };
  const int npig = npig_arr[k * kA + a];
  if (npig == 0) {
    for (int r = tid; r < kR; r += NT) precision[prec_at(r)] = -1.0;
    if (tid == 0) recall[rec_at] = -1.0;
    return;
  }
  for (int r = tid; r < kR; r += NT) q[r] = 0.0;
  const long long cs = cstart[k], ce = cend[k], nd = ce - cs;
  const double npd = (double)npig, eps = 2.220446049250313080847263336181640625e-16;   // np.spacing(1)
  auto flag = [&](long long d) {                          // -1 outside the sequence, 0 ignored, 1 TP, 2 FP
    const unsigned long long x = g0[d];
    if ((long long)(x >> kPosShift) >= maxdet) return -1;
    if ((x >> pair) & 1ull) return 1;
    return ((g1[d] >> pair) & 1ull) ? 0 : 2;
  };
  auto count = [](int f) { return f == 1 ? (1ull << 32) : f == 2 ? 1ull : 0ull; };
  unsigned long long loc = 0;
  for (long long d = cs + tid; d < ce; d += NT) loc += count(flag(d));
  unsigned long long totals;
  voc::block_exclusive_scan<unsigned long long, voc::AddOp, NT>(loc, 0ull, voc::AddOp(), smc, &totals);
  const long long TT = (long long)(totals >> 32), TF = (long long)(totals & 0xffffffffull);
  __syncthreads();                                        // q zeroed before any lookup writes it
  unsigned long long carry_cnt = 0;
  double carry_max = 0.0;
  for (long long q0 = 0; q0 < nd; q0 += CH) {
    int f[IT];
    unsigned long long mine = 0;
#pragma unroll
    for (int i = 0; i < IT; ++i) {
      const long long p = q0 + (long long)tid * IT + i;
      f[i] = p < nd ? flag(ce - 1 - p) : -1;
      mine += count(f[i]);
    }
    unsigned long long chunk_cnt;
    unsigned long long after = carry_cnt + voc::block_exclusive_scan<unsigned long long, voc::AddOp, NT>(
                                               mine, 0ull, voc::AddOp(), smc, &chunk_cnt);
    double pr[IT], lmax[IT];
    long long tpc[IT];
    double run = 0.0;
#pragma unroll
    for (int i = 0; i < IT; ++i) {
      const long long tp = TT - (long long)(after >> 32), fp = TF - (long long)(after & 0xffffffffull);
      tpc[i] = tp;
      pr[i] = f[i] < 0 ? 0.0 : __ddiv_rn((double)tp, __dadd_rn((double)(fp + tp), eps));
      run = fmax(run, pr[i]);
      lmax[i] = run;
      after += count(f[i]);
    }
    double chunk_max;
    const double before_max = fmax(carry_max, voc::block_exclusive_scan<double, voc::MaxOp, NT>(
                                                  run, 0.0, voc::MaxOp(), smd, &chunk_max));
#pragma unroll
    for (int i = 0; i < IT; ++i) {
      if (f[i] != 1) continue;
      const double env = fmax(before_max, lmax[i]);
      const double rc = __ddiv_rn((double)tpc[i], npd), rc_prev = __ddiv_rn((double)(tpc[i] - 1), npd);
      for (int r = 0; r < kR; ++r)
        if (rc_prev < thr.rec[r] && thr.rec[r] <= rc) q[r] = env;
    }
    carry_cnt += chunk_cnt;
    carry_max = fmax(carry_max, chunk_max);
  }
  __syncthreads();
  for (int r = tid; r < kR; r += NT) precision[prec_at(r)] = thr.rec[r] <= 0.0 ? carry_max : q[r];
  if (tid == 0) recall[rec_at] = __ddiv_rn((double)TT, npd);
}

// ---- workspace ----------------------------------------------------------------------------------------------------
struct EvalWorkspace {
  uint32_t *ka, *va, *kb, *vb, *ckey, *corder, *hist, *sums;
  int *cell_begin, *cell_end, *npig, *cstart, *cend;
  unsigned long long *m0, *m1, *g0, *g1;
  double* iou;
  uint8_t* gtm;
  long long ntiles;
};

// Carves the workspace; returns the bytes needed (base == nullptr: size query only).
inline int64_t eval_workspace(void* base, long long n, long long cells, int K, long long n_gt, EvalWorkspace* ws) {
  const long long ntiles = (n + voc::kSortTile - 1) / voc::kSortTile;
  const long long hist_len = (long long)voc::kRadixBins * ntiles;
  char* p = static_cast<char*>(base);
  int64_t off = 0;
  auto take = [&](int64_t bytes) {
    char* r = p ? p + off : nullptr;
    off += round_up64(bytes > 0 ? bytes : 1, 256);
    return r;
  };
  EvalWorkspace w{};
  w.ntiles = ntiles;
  w.ka = reinterpret_cast<uint32_t*>(take(4 * n));
  w.va = reinterpret_cast<uint32_t*>(take(4 * n));
  w.kb = reinterpret_cast<uint32_t*>(take(4 * n));
  w.vb = reinterpret_cast<uint32_t*>(take(4 * n));
  w.ckey = reinterpret_cast<uint32_t*>(take(4 * n));
  w.corder = reinterpret_cast<uint32_t*>(take(4 * n));
  w.hist = reinterpret_cast<uint32_t*>(take(4 * hist_len));
  w.sums = reinterpret_cast<uint32_t*>(take(4 * voc::scan_sums_len(hist_len)));
  w.cell_begin = reinterpret_cast<int*>(take(4 * cells));
  w.cell_end = reinterpret_cast<int*>(take(4 * cells));
  w.npig = reinterpret_cast<int*>(take(4 * (int64_t)K * kA));
  w.cstart = reinterpret_cast<int*>(take(4 * (int64_t)K));
  w.cend = reinterpret_cast<int*>(take(4 * (int64_t)K));
  w.m0 = reinterpret_cast<unsigned long long*>(take(8 * n));
  w.m1 = reinterpret_cast<unsigned long long*>(take(8 * n));
  w.g0 = reinterpret_cast<unsigned long long*>(take(8 * n));
  w.g1 = reinterpret_cast<unsigned long long*>(take(8 * n));
  w.iou = reinterpret_cast<double*>(take(8 * (int64_t)kMaxDet * n_gt));
  w.gtm = reinterpret_cast<uint8_t*>(take((int64_t)kPairs * n_gt));
  if (ws) *ws = w;
  return off;
}

inline int key_bits(long long maxkey) {
  int bits = 0;
  while (bits < 32 && (maxkey >> bits)) ++bits;
  return bits;
}

// Stable LSD passes (voc::radix_hist_kernel / radix_scatter_kernel, 8-bit digits) over the low `bits` bits of
// (k, v); the result is left in (k, v), the other pair is scratch.
inline void radix_passes(uint32_t*& k, uint32_t*& v, uint32_t*& kt, uint32_t*& vt, long long n, int bits,
                         const EvalWorkspace& w, cudaStream_t st) {
  for (int shift = 0; shift < bits; shift += 8) {
    voc::radix_hist_kernel<<<(unsigned)w.ntiles, voc::kSortNT, 0, st>>>(k, n, shift, w.hist, (int)w.ntiles);
    YNB_COUNT_LAUNCH();
    voc::launch_scan_u32(w.hist, (long long)voc::kRadixBins * w.ntiles, w.sums, st);
    voc::radix_scatter_kernel<<<(unsigned)w.ntiles, voc::kSortNT, 0, st>>>(k, v, n, shift, w.hist, (int)w.ntiles,
                                                                           kt, vt);
    YNB_COUNT_LAUNCH();
    std::swap(k, kt);
    std::swap(v, vt);
  }
}

inline cudaError_t launch_coco_eval(const int* rows, long long n, int num_classes, int num_images,
                                    const int* image_rank, const int* class_cat, int K, const double* gt_boxes,
                                    const double* gt_area, const uint8_t* gt_crowd, const int* gt_start,
                                    long long n_gt, const Thresholds& thr, double* precision, double* recall,
                                    const EvalWorkspace& w, cudaStream_t st) {
  cudaError_t r;
  const long long cells = (long long)num_images * K;
  if ((r = cudaMemsetAsync(w.npig, 0, sizeof(int) * K * kA, st)) != cudaSuccess) return r;
  if ((r = cudaMemsetAsync(w.cstart, 0, sizeof(int) * K, st)) != cudaSuccess) return r;
  if ((r = cudaMemsetAsync(w.cend, 0, sizeof(int) * K, st)) != cudaSuccess) return r;
  if (cells > 0 && (r = cudaMemsetAsync(w.cell_begin, 0, sizeof(int) * cells, st)) != cudaSuccess) return r;
  if (cells > 0 && (r = cudaMemsetAsync(w.cell_end, 0, sizeof(int) * cells, st)) != cudaSuccess) return r;
  if (n_gt > 0 && (r = cudaMemsetAsync(w.gtm, 0, (size_t)kPairs * n_gt, st)) != cudaSuccess) return r;
  if (n > 0) {
    // 1. cell order: score, then cell
    uint32_t *k = w.ka, *v = w.va, *kt = w.kb, *vt = w.vb;
    coco_score_keys_kernel<<<voc::blocks_for(n, 256), 256, 0, st>>>(rows, nullptr, n, k, v);
    YNB_COUNT_LAUNCH();
    radix_passes(k, v, kt, vt, n, 32, w, st);
    coco_cell_keys_kernel<<<voc::blocks_for(n, 256), 256, 0, st>>>(rows, v, n, image_rank, num_images, class_cat,
                                                                    num_classes, K, k);
    YNB_COUNT_LAUNCH();
    radix_passes(k, v, kt, vt, n, key_bits(cells), w, st);
    if ((r = cudaMemcpyAsync(w.ckey, k, 4 * n, cudaMemcpyDeviceToDevice, st)) != cudaSuccess) return r;
    if ((r = cudaMemcpyAsync(w.corder, v, 4 * n, cudaMemcpyDeviceToDevice, st)) != cudaSuccess) return r;
    coco_cell_bounds_kernel<<<voc::blocks_for(n, 256), 256, 0, st>>>(w.ckey, n, cells, w.cell_begin, w.cell_end);
    YNB_COUNT_LAUNCH();
  }
  // 2. evaluateImg per cell (cells with GT only still count towards npig)
  if (cells > 0) {
    coco_match_kernel<<<(unsigned)cells, kMatchNT, 0, st>>>(rows, w.corder, w.cell_begin, w.cell_end, K, gt_boxes,
                                                            gt_area, gt_crowd, gt_start, n_gt, thr, w.iou, w.gtm,
                                                            w.m0, w.m1, w.npig);
    YNB_COUNT_LAUNCH();
  }
  if (n > 0) {
    // 3. per-category order over the cell order: score, then category (cut detections last)
    uint32_t *k = w.ka, *v = w.va, *kt = w.kb, *vt = w.vb;
    coco_score_keys_kernel<<<voc::blocks_for(n, 256), 256, 0, st>>>(rows, w.corder, n, k, v);
    YNB_COUNT_LAUNCH();
    radix_passes(k, v, kt, vt, n, 32, w, st);
    coco_cat_keys_kernel<<<voc::blocks_for(n, 256), 256, 0, st>>>(w.ckey, w.cell_begin, v, n, cells, K, k);
    YNB_COUNT_LAUNCH();
    radix_passes(k, v, kt, vt, n, key_bits(K), w, st);
    coco_cat_gather_kernel<<<voc::blocks_for(n, 256), 256, 0, st>>>(k, v, n, K, w.m0, w.m1, w.g0, w.g1, w.cstart,
                                                                    w.cend);
    YNB_COUNT_LAUNCH();
  }
  // 4. accumulate
  coco_accumulate_kernel<<<(unsigned)(K * kA * kM * kT), voc::kApNT, 0, st>>>(w.g0, w.g1, w.cstart, w.cend, w.npig,
                                                                               K, thr, precision, recall);
  YNB_COUNT_LAUNCH();
  return cudaGetLastError();
}

}  // namespace coco
}  // namespace ynb
