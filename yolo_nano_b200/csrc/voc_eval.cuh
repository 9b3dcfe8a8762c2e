// VOC07 mAP on the device: the evaluators' det-file round trip and voc_eval (evaluator/vocapi_evaluator.py,
// ssd.pytorch lineage: no +1 pixel in the overlaps, ap = -1 for a class without detection lines).
//
//   append    engine rows after map_boxes -> one compact int32 row per detection line, in file order
//             (image, kept row): [image, class, milli, x1, y1, x2, y2].  milli = the integer of '{:.3f}' of the
//             score, xk = the integer of '{:.1f}' of (box_k + 1) with the +1 in float32; both rounded half-even on
//             the exact binary value, as Python's formatting does.  float('n.nnn') == n / 1000.0 and
//             float('n.n') == n / 10.0 in IEEE double, so the rows carry exactly what voc_eval parses back.
//             A '-0.0' box field (values in (-0.05, 0] after the +1) is stored as INT32_MIN.
//   evaluate  stable LSD radix sort by (class, 1000 - milli): ties stay in file order, the order NMS defines for
//             its own ties; overlaps / argmax against the image's GT of that class; first-claim resolution; per
//             class tp / fp scans and the AP.  Every float64 expression is written with explicit _rn intrinsics:
//             the build contracts a*b+c into FMA otherwise, and the 07 AP is bit-identical to NumPy's.
//
// The greedy matching of voc_eval is order-independent once ovmax / jmax are known (they do not depend on which GT
// are claimed): a detection with ovmax > thr on a non-difficult jmax is TP exactly when it is the first in sorted
// order among the detections aiming at the same GT.  That is an atomicMin of the sorted position per GT.
#pragma once
#include <cuda_runtime.h>
#include <float.h>
#include <stdint.h>

#include <utility>

#include "common.cuh"

namespace ynb {
namespace voc {

constexpr int kRowInts = 7;
constexpr int kScoreBins = 1001;            // milli in [0, 1000]
constexpr int kFlagIgnored = 0, kFlagTP = 1, kFlagFP = 2;
constexpr int kCandFP = -1, kCandIgnored = -2;

// ---- decimal fields ---------------------------------------------------------------------------------------------
// round_half_even(|x| * 10^digits) of the exact float32 value, in integer arithmetic on the mantissa.  Returns false
// when x is not finite or the integer does not fit an int32.
__device__ __forceinline__ bool decimal_magnitude(float x, uint64_t pow10, uint64_t* q_out) {
  const uint32_t u = __float_as_uint(x);
  const uint32_t ex = (u >> 23) & 0xffu, fr = u & 0x7fffffu;
  if (ex == 0xffu) return false;
  const uint64_t m = ex ? (fr | 0x800000u) : fr;           // x = m * 2^e
  const int e = ex ? (int)ex - 150 : -149;
  const uint64_t big = m * pow10;                          // < 2^34
  uint64_t q;
  if (e >= 0) {
    if (e > 30 || big > ((uint64_t)INT32_MAX >> e)) return false;
    q = big << e;
  } else if (-e >= 40) {
    q = 0;                                                 // big / 2^40 < 2^-6: rounds to 0
  } else {
    const int s = -e;
    q = big >> s;
    const uint64_t rem = big & ((1ull << s) - 1), half = 1ull << (s - 1);
    if (rem > half || (rem == half && (q & 1))) ++q;
  }
  if (q > (uint64_t)INT32_MAX) return false;
  *q_out = q;
  return true;
}

__device__ __forceinline__ double tenths_value(int32_t n) {
  return n == INT32_MIN ? -0.0 : __ddiv_rn((double)n, 10.0);
}

// ---- block scans --------------------------------------------------------------------------------------------------
template <typename T, typename Op, int NT>
__device__ __forceinline__ T block_exclusive_scan(T v, T identity, Op op, T* sm /* [NT / 32] */, T* total) {
  constexpr int NW = NT / 32;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  T incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const T y = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl = op(y, incl);
  }
  if (lane == 31) sm[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    T w = lane < NW ? sm[lane] : identity;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const T y = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w = op(y, w);
    }
    if (lane < NW) sm[lane] = w;
  }
  __syncthreads();
  T excl = __shfl_up_sync(0xffffffffu, incl, 1);
  if (lane == 0) excl = identity;
  if (warp > 0) excl = op(sm[warp - 1], excl);
  *total = sm[NW - 1];
  __syncthreads();
  return excl;
}

struct AddOp {
  template <typename T>
  __device__ __forceinline__ T operator()(T a, T b) const { return a + b; }
};
struct MaxOp {
  __device__ __forceinline__ double operator()(double a, double b) const { return fmax(a, b); }
};

// ---- append -------------------------------------------------------------------------------------------------------
// One block per image: its first slot is state[0] + sum(counts[0..b)) (a prefix sum, so arena order == file order).
__global__ void __launch_bounds__(256)
voc_append_kernel(const float* __restrict__ boxes, const float* __restrict__ scores, const int* __restrict__ cls,
                  const int* __restrict__ counts, int batch, long long n_per_image, int image_base, int num_classes,
                  int* __restrict__ rows, long long capacity, long long* __restrict__ state) {
  __shared__ long long sm[8];
  const int b = blockIdx.x;
  long long before = 0;
  for (int i = threadIdx.x; i < b; i += blockDim.x) before += min((long long)max(counts[i], 0), n_per_image);
  long long tot;
  block_exclusive_scan<long long, AddOp, 256>(before, 0ll, AddOp(), sm, &tot);
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
    uint64_t q = 0;
    const float s = scores[src];
    ok = decimal_magnitude(s, 1000, &q) && ok;
    if (s < 0.0f && q != 0) ok = false;                    // negative scores do not sort on the 1001 bins
    if (q > 1000) { ok = false; q = 1000; }
    row[2] = (int)q;
    for (int j = 0; j < 4; ++j) {
      const float v = __fadd_rn(boxes[src * 4 + j], 1.0f);  // dets[k, j] + 1 on a float32 array
      uint64_t t = 0;
      ok = decimal_magnitude(v, 10, &t) && ok;
      const bool neg = __float_as_uint(v) >> 31;
      row[3 + j] = neg ? (t ? -(int)t : INT32_MIN) : (int)t;
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

// Runs after voc_append_kernel on the same stream: the row total moves on only once every block has read it.
__global__ void __launch_bounds__(256)
voc_append_total_kernel(const int* __restrict__ counts, int batch, long long n_per_image, long long* state) {
  __shared__ long long sm[8];
  long long s = 0;
  for (int i = threadIdx.x; i < batch; i += blockDim.x) s += min((long long)max(counts[i], 0), n_per_image);
  long long tot;
  block_exclusive_scan<long long, AddOp, 256>(s, 0ll, AddOp(), sm, &tot);
  if (threadIdx.x == 0) state[0] += tot;
}

inline cudaError_t launch_voc_append(const float* boxes, const float* scores, const int* cls, const int* counts,
                                     int batch, long long n_per_image, int image_base, int num_classes, int* rows,
                                     long long capacity, long long* state, cudaStream_t st) {
  voc_append_kernel<<<batch, 256, 0, st>>>(boxes, scores, cls, counts, batch, n_per_image, image_base, num_classes,
                                           rows, capacity, state);
  YNB_COUNT_LAUNCH();
  voc_append_total_kernel<<<1, 256, 0, st>>>(counts, batch, n_per_image, state);
  YNB_COUNT_LAUNCH();
  return cudaGetLastError();
}

// ---- device-wide exclusive scan of uint32 (in place) --------------------------------------------------------------
constexpr int kScanNT = 1024, kScanIT = 4, kScanTile = kScanNT * kScanIT;

__global__ void __launch_bounds__(kScanNT) scan_tiles_kernel(uint32_t* __restrict__ a, long long n,
                                                             uint32_t* __restrict__ sums) {
  __shared__ uint32_t sm[kScanNT / 32];
  const long long base = (long long)blockIdx.x * kScanTile + (long long)threadIdx.x * kScanIT;
  uint32_t v[kScanIT], s = 0;
#pragma unroll
  for (int i = 0; i < kScanIT; ++i) {
    v[i] = base + i < n ? a[base + i] : 0u;
    s += v[i];
  }
  uint32_t tot;
  uint32_t run = block_exclusive_scan<uint32_t, AddOp, kScanNT>(s, 0u, AddOp(), sm, &tot);
#pragma unroll
  for (int i = 0; i < kScanIT; ++i) {
    if (base + i < n) a[base + i] = run;
    run += v[i];
  }
  if (threadIdx.x == 0) sums[blockIdx.x] = tot;
}

// One block, serial over chunks with a carry: the tile sums are few (n / 4096).
__global__ void __launch_bounds__(kScanNT) scan_sums_kernel(uint32_t* __restrict__ sums, int n) {
  __shared__ uint32_t sm[kScanNT / 32];
  uint32_t carry = 0;
  for (int c0 = 0; c0 < n; c0 += kScanNT) {
    const int i = c0 + threadIdx.x;
    const uint32_t v = i < n ? sums[i] : 0u;
    uint32_t tot;
    const uint32_t e = block_exclusive_scan<uint32_t, AddOp, kScanNT>(v, 0u, AddOp(), sm, &tot);
    if (i < n) sums[i] = carry + e;
    carry += tot;
  }
}

__global__ void __launch_bounds__(256) scan_add_kernel(uint32_t* __restrict__ a, long long n,
                                                       const uint32_t* __restrict__ sums) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) a[i] += sums[i / kScanTile];
}

inline long long scan_sums_len(long long n) { return (n + kScanTile - 1) / kScanTile; }

inline void launch_scan_u32(uint32_t* a, long long n, uint32_t* sums, cudaStream_t st) {
  const long long nt = scan_sums_len(n);
  if (nt == 0) return;
  scan_tiles_kernel<<<(unsigned)nt, kScanNT, 0, st>>>(a, n, sums);
  YNB_COUNT_LAUNCH();
  if (nt > 1) {
    scan_sums_kernel<<<1, kScanNT, 0, st>>>(sums, (int)nt);
    YNB_COUNT_LAUNCH();
    scan_add_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(a, n, sums);
    YNB_COUNT_LAUNCH();
  }
}

// ---- stable LSD radix sort of (key, arena index) ------------------------------------------------------------------
// 8-bit digits.  A tile of 4096 is ordered by (digit, position in tile) with a bitonic network in shared memory, so
// the scatter keeps input order among equal digits; tiles are placed digit-major, tile-minor by the scanned counts.
constexpr int kSortNT = 256, kSortTile = 4096, kRadixBins = 256;

__global__ void voc_sort_init_kernel(const int* __restrict__ rows, long long n, int num_classes,
                                     uint32_t* __restrict__ keys, uint32_t* __restrict__ vals) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int* r = rows + (size_t)i * kRowInts;
  const int c = min(max(r[1], 0), num_classes - 1), milli = min(max(r[2], 0), 1000);
  keys[i] = (uint32_t)(c * kScoreBins + (1000 - milli));
  vals[i] = (uint32_t)i;
}

__global__ void __launch_bounds__(kSortNT)
radix_hist_kernel(const uint32_t* __restrict__ keys, long long n, int shift, uint32_t* __restrict__ hist, int ntiles) {
  __shared__ uint32_t h[kRadixBins];
  for (int i = threadIdx.x; i < kRadixBins; i += kSortNT) h[i] = 0;
  __syncthreads();
  const long long base = (long long)blockIdx.x * kSortTile;
  for (int i = threadIdx.x; i < kSortTile; i += kSortNT)
    if (base + i < n) atomicAdd(&h[(keys[base + i] >> shift) & 0xffu], 1u);
  __syncthreads();
  for (int i = threadIdx.x; i < kRadixBins; i += kSortNT) hist[(size_t)i * ntiles + blockIdx.x] = h[i];
}

__global__ void __launch_bounds__(kSortNT)
radix_scatter_kernel(const uint32_t* __restrict__ kin, const uint32_t* __restrict__ vin, long long n, int shift,
                     const uint32_t* __restrict__ offs, int ntiles, uint32_t* __restrict__ kout,
                     uint32_t* __restrict__ vout) {
  __shared__ uint32_t s[kSortTile];
  __shared__ uint32_t start[kRadixBins];
  const long long base = (long long)blockIdx.x * kSortTile;
  const int cnt = (int)min((long long)kSortTile, n - base);
  for (int i = threadIdx.x; i < kSortTile; i += kSortNT)
    s[i] = i < cnt ? ((((kin[base + i] >> shift) & 0xffu) << 12) | (uint32_t)i) : 0xffffffffu;
  __syncthreads();
  for (int k = 2; k <= kSortTile; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int p = threadIdx.x; p < kSortTile / 2; p += kSortNT) {
        const int i = ((p & ~(j - 1)) << 1) | (p & (j - 1)), l = i + j;
        const uint32_t a = s[i], b = s[l];
        if ((a > b) == ((i & k) == 0)) { s[i] = b; s[l] = a; }
      }
      __syncthreads();
    }
  }
  for (int p = threadIdx.x; p < cnt; p += kSortNT) {
    const uint32_t d = s[p] >> 12;
    if (p == 0 || (s[p - 1] >> 12) != d) start[d] = p;
  }
  __syncthreads();
  for (int p = threadIdx.x; p < cnt; p += kSortNT) {
    const uint32_t d = s[p] >> 12, loc = s[p] & 0xfffu;
    const size_t dst = (size_t)offs[(size_t)d * ntiles + blockIdx.x] + (p - start[d]);
    kout[dst] = kin[base + loc];
    vout[dst] = vin[base + loc];
  }
}

// ---- matching -----------------------------------------------------------------------------------------------------
// Per sorted detection d: ovmax / jmax over ALL GT of its (image, class) bucket, difficult ones included (np.max
// propagates NaN, np.argmax takes the first maximum or the first NaN), then the candidate GT slot, FP or ignored.
__global__ void __launch_bounds__(256)
voc_match_kernel(const int* __restrict__ rows, const uint32_t* __restrict__ order, long long n, int num_classes,
                 int num_images, const double* __restrict__ gt_boxes, const uint8_t* __restrict__ gt_difficult,
                 const int* __restrict__ gt_start, double ovthresh, int* __restrict__ cand, int* __restrict__ claim) {
  const long long d = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= n) return;
  const int* r = rows + (size_t)order[d] * kRowInts;
  const int img = r[0], c = r[1];
  const double b0 = tenths_value(r[3]), b1 = tenths_value(r[4]), b2 = tenths_value(r[5]), b3 = tenths_value(r[6]);
  int gs = 0, ge = 0;
  if (img >= 0 && img < num_images && c >= 0 && c < num_classes) {
    gs = gt_start[(size_t)img * num_classes + c];
    ge = gt_start[(size_t)img * num_classes + c + 1];
  }
  const double barea = __dmul_rn(__dsub_rn(b2, b0), __dsub_rn(b3, b1));
  double ovmax = -INFINITY;
  int jmax = -1;
  for (int j = gs; j < ge; ++j) {
    const double g0 = gt_boxes[4 * j], g1 = gt_boxes[4 * j + 1], g2 = gt_boxes[4 * j + 2], g3 = gt_boxes[4 * j + 3];
    const double iw = fmax(__dsub_rn(fmin(g2, b2), fmax(g0, b0)), 0.0);
    const double ih = fmax(__dsub_rn(fmin(g3, b3), fmax(g1, b1)), 0.0);
    const double inters = __dmul_rn(iw, ih);
    const double uni = __dsub_rn(__dadd_rn(barea, __dmul_rn(__dsub_rn(g2, g0), __dsub_rn(g3, g1))), inters);
    const double ov = __ddiv_rn(inters, uni);
    if (isnan(ov)) { ovmax = ov; jmax = j; break; }
    if (jmax < 0 || ov > ovmax) { ovmax = ov; jmax = j; }
  }
  int cd = kCandFP;
  if (ovmax > ovthresh) {
    if (gt_difficult[jmax]) {
      cd = kCandIgnored;
    } else {
      cd = jmax;
      atomicMin(claim + jmax, (int)d);
    }
  }
  cand[d] = cd;
}

// TP = first claimant of its GT; class ranges [cstart, cend) of the sorted order (zeroed before: empty classes).
__global__ void __launch_bounds__(256)
voc_resolve_kernel(const uint32_t* __restrict__ keys, long long n, const int* __restrict__ cand,
                   const int* __restrict__ claim, int8_t* __restrict__ flags, int* __restrict__ cstart,
                   int* __restrict__ cend) {
  const long long d = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= n) return;
  const int cd = cand[d];
  flags[d] = (int8_t)(cd == kCandIgnored ? kFlagIgnored : (cd >= 0 && claim[cd] == (int)d) ? kFlagTP : kFlagFP);
  const uint32_t c = keys[d] / kScoreBins;
  if (d == 0 || keys[d - 1] / kScoreBins != c) cstart[c] = (int)d;
  if (d == n - 1 || keys[d + 1] / kScoreBins != c) cend[c] = (int)d + 1;
}

__global__ void __launch_bounds__(256)
voc_npos_kernel(const uint8_t* __restrict__ gt_difficult, const int* __restrict__ gt_start, int num_images,
                int num_classes, int* __restrict__ npos) {
  const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= (long long)num_images * num_classes) return;
  int k = 0;
  for (int j = gt_start[b]; j < gt_start[b + 1]; ++j) k += !gt_difficult[j];
  if (k) atomicAdd(npos + (b % num_classes), k);
}

// ---- per-class AP -------------------------------------------------------------------------------------------------
// One block per class walks its sorted range from the END in chunks: with the class totals known, the cumsums at d
// are total - (count after d), and the precision envelope max(prec[d..]) is a forward max-scan in that walk order.
//   rec[d] = tp / npos,  prec[d] = tp / max(tp + fp, eps64)
//   07:   p_i = envelope at the first d with rec[d] >= i * 0.1 (rec is non-decreasing), 0 if none;
//         ap = sum_i p_i / 11 in order i = 0..10
//   area: sum over TPs d of (rec[d] - rec[d-1]) * envelope[d]  (the recall change points of voc_ap; the closing
//         (1 - rec) * 0 term adds +0), reduced in a fixed order; NaN when npos == 0, as NumPy gives.
constexpr int kApNT = 512, kApIT = 8, kApChunk = kApNT * kApIT;

__global__ void __launch_bounds__(kApNT)
voc_class_ap_kernel(const int8_t* __restrict__ flags, const int* __restrict__ cstart, const int* __restrict__ cend,
                    const int* __restrict__ npos_arr, int use_07, double* __restrict__ ap_out) {
  __shared__ unsigned long long smc[kApNT / 32];
  __shared__ double smd[kApNT / 32];
  __shared__ double p07[11];
  __shared__ double red[kApNT];
  const int c = blockIdx.x, t = threadIdx.x;
  const long long cs = cstart[c], ce = cend[c], nd = ce - cs;
  if (nd <= 0) {
    if (t == 0) ap_out[c] = -1.0;
    return;
  }
  if (t < 11) p07[t] = 0.0;
  const int npos = npos_arr[c];
  const double npd = (double)npos;
  // class totals (tp << 32 | fp)
  unsigned long long loc = 0;
  for (long long d = cs + t; d < ce; d += kApNT) {
    const int f = flags[d];
    loc += f == kFlagTP ? (1ull << 32) : f == kFlagFP ? 1ull : 0ull;
  }
  unsigned long long totals;
  block_exclusive_scan<unsigned long long, AddOp, kApNT>(loc, 0ull, AddOp(), smc, &totals);
  const long long TT = (long long)(totals >> 32), TF = (long long)(totals & 0xffffffffull);
  unsigned long long carry_cnt = 0;
  double carry_max = 0.0, area = 0.0;
  for (long long q0 = 0; q0 < nd; q0 += kApChunk) {
    int f[kApIT];
    unsigned long long mine = 0;
#pragma unroll
    for (int i = 0; i < kApIT; ++i) {
      const long long q = q0 + (long long)t * kApIT + i;
      f[i] = q < nd ? flags[ce - 1 - q] : -1;
      mine += f[i] == kFlagTP ? (1ull << 32) : f[i] == kFlagFP ? 1ull : 0ull;
    }
    unsigned long long chunk_cnt;
    unsigned long long after = carry_cnt + block_exclusive_scan<unsigned long long, AddOp, kApNT>(
                                               mine, 0ull, AddOp(), smc, &chunk_cnt);
    double prec[kApIT], lmax[kApIT];
    long long tpc[kApIT];
    double run = 0.0;
#pragma unroll
    for (int i = 0; i < kApIT; ++i) {
      const long long tp = TT - (long long)(after >> 32), fp = TF - (long long)(after & 0xffffffffull);
      tpc[i] = tp;
      const long long den = tp + fp;
      prec[i] = f[i] < 0 ? 0.0 : __ddiv_rn((double)tp, den > 0 ? (double)den : DBL_EPSILON);
      run = fmax(run, prec[i]);
      lmax[i] = run;
      after += f[i] == kFlagTP ? (1ull << 32) : f[i] == kFlagFP ? 1ull : 0ull;
    }
    double chunk_max;
    const double before_max = fmax(carry_max, block_exclusive_scan<double, MaxOp, kApNT>(run, 0.0, MaxOp(), smd,
                                                                                          &chunk_max));
#pragma unroll
    for (int i = 0; i < kApIT; ++i) {
      if (f[i] < 0) continue;
      const long long d = ce - 1 - (q0 + (long long)t * kApIT + i);
      const double env = fmax(before_max, lmax[i]);
      const double rec = __ddiv_rn((double)tpc[i], npd);
      const double rec_prev = __ddiv_rn((double)(tpc[i] - (f[i] == kFlagTP)), npd);
      if (f[i] == kFlagTP) area = __dadd_rn(area, __dmul_rn(__dsub_rn(rec, rec_prev), env));
      for (int k = 0; k < 11; ++k) {
        const double thr = __dmul_rn((double)k, 0.1);
        if (rec >= thr && (d == cs || rec_prev < thr)) p07[k] = env;
      }
    }
    carry_cnt += chunk_cnt;
    carry_max = fmax(carry_max, chunk_max);
  }
  red[t] = area;
  __syncthreads();
  for (int s = kApNT / 2; s > 0; s >>= 1) {
    if (t < s) red[t] = __dadd_rn(red[t], red[t + s]);
    __syncthreads();
  }
  if (t == 0) {
    double ap;
    if (use_07) {
      ap = 0.0;
      for (int k = 0; k < 11; ++k) ap = __dadd_rn(ap, __ddiv_rn(p07[k], 11.0));
    } else {
      ap = npos == 0 ? __longlong_as_double(0x7ff8000000000000ll) : red[0];
    }
    ap_out[c] = ap;
  }
}

// ---- workspace ----------------------------------------------------------------------------------------------------
struct EvalWorkspace {
  uint32_t *k0, *v0, *k1, *v1, *hist, *sums;
  int *cand, *claim, *cstart, *cend;
  int8_t* flags;
  long long ntiles;
};

inline int radix_passes(int num_classes) {
  const uint32_t maxkey = (uint32_t)num_classes * kScoreBins - 1;
  int bits = 1;
  while (bits < 32 && (maxkey >> bits)) ++bits;
  return (bits + 7) / 8;
}

// Carves the workspace; returns the bytes needed (ws == nullptr: size query only).
inline int64_t eval_workspace(void* base, long long n, int num_classes, long long n_gt, EvalWorkspace* ws) {
  const long long ntiles = (n + kSortTile - 1) / kSortTile;
  const long long hist_len = (long long)kRadixBins * ntiles;
  char* p = static_cast<char*>(base);
  int64_t off = 0;
  auto take = [&](int64_t bytes) {
    char* r = p ? p + off : nullptr;
    off += round_up64(bytes > 0 ? bytes : 1, 256);
    return r;
  };
  EvalWorkspace w{};
  w.ntiles = ntiles;
  w.k0 = reinterpret_cast<uint32_t*>(take(4 * n));
  w.v0 = reinterpret_cast<uint32_t*>(take(4 * n));
  w.k1 = reinterpret_cast<uint32_t*>(take(4 * n));
  w.v1 = reinterpret_cast<uint32_t*>(take(4 * n));
  w.hist = reinterpret_cast<uint32_t*>(take(4 * hist_len));
  w.sums = reinterpret_cast<uint32_t*>(take(4 * scan_sums_len(hist_len)));
  w.cand = reinterpret_cast<int*>(take(4 * n));
  w.claim = reinterpret_cast<int*>(take(4 * n_gt));
  w.cstart = reinterpret_cast<int*>(take(4 * num_classes));
  w.cend = reinterpret_cast<int*>(take(4 * num_classes));
  w.flags = reinterpret_cast<int8_t*>(take(n));
  if (ws) *ws = w;
  return off;
}

inline unsigned blocks_for(long long n, int nt) { return (unsigned)((n + nt - 1) / nt); }

// Sorted order -> order_out (arena index per sorted position) when requested; flags_out likewise.
inline cudaError_t launch_voc_eval(const int* rows, long long n, int num_classes, int num_images,
                                   const double* gt_boxes, const uint8_t* gt_difficult, const int* gt_start,
                                   long long n_gt, double ovthresh, int use_07, double* ap, int* npos,
                                   int* order_out, int8_t* flags_out, const EvalWorkspace& w, cudaStream_t st) {
  cudaError_t r;
  if ((r = cudaMemsetAsync(npos, 0, sizeof(int) * num_classes, st)) != cudaSuccess) return r;
  if ((long long)num_images * num_classes > 0) {
    voc_npos_kernel<<<blocks_for((long long)num_images * num_classes, 256), 256, 0, st>>>(
        gt_difficult, gt_start, num_images, num_classes, npos);
    YNB_COUNT_LAUNCH();
  }
  if ((r = cudaMemsetAsync(w.cstart, 0, sizeof(int) * num_classes, st)) != cudaSuccess) return r;
  if ((r = cudaMemsetAsync(w.cend, 0, sizeof(int) * num_classes, st)) != cudaSuccess) return r;
  const uint32_t* order = w.v0;
  const uint32_t* keys = w.k0;
  if (n > 0) {
    voc_sort_init_kernel<<<blocks_for(n, 256), 256, 0, st>>>(rows, n, num_classes, w.k0, w.v0);
    YNB_COUNT_LAUNCH();
    uint32_t *kin = w.k0, *vin = w.v0, *kout = w.k1, *vout = w.v1;
    const int passes = radix_passes(num_classes);
    for (int ps = 0; ps < passes; ++ps) {
      radix_hist_kernel<<<(unsigned)w.ntiles, kSortNT, 0, st>>>(kin, n, 8 * ps, w.hist, (int)w.ntiles);
      YNB_COUNT_LAUNCH();
      launch_scan_u32(w.hist, (long long)kRadixBins * w.ntiles, w.sums, st);
      radix_scatter_kernel<<<(unsigned)w.ntiles, kSortNT, 0, st>>>(kin, vin, n, 8 * ps, w.hist, (int)w.ntiles,
                                                                   kout, vout);
      YNB_COUNT_LAUNCH();
      std::swap(kin, kout);
      std::swap(vin, vout);
    }
    keys = kin;
    order = vin;
    if (n_gt > 0 && (r = cudaMemsetAsync(w.claim, 0x7f, sizeof(int) * n_gt, st)) != cudaSuccess) return r;
    voc_match_kernel<<<blocks_for(n, 256), 256, 0, st>>>(rows, order, n, num_classes, num_images, gt_boxes,
                                                         gt_difficult, gt_start, ovthresh, w.cand, w.claim);
    YNB_COUNT_LAUNCH();
    voc_resolve_kernel<<<blocks_for(n, 256), 256, 0, st>>>(keys, n, w.cand, w.claim, w.flags, w.cstart, w.cend);
    YNB_COUNT_LAUNCH();
  }
  voc_class_ap_kernel<<<num_classes, kApNT, 0, st>>>(w.flags, w.cstart, w.cend, npos, use_07, ap);
  YNB_COUNT_LAUNCH();
  if (n > 0 && order_out &&
      (r = cudaMemcpyAsync(order_out, order, sizeof(int) * n, cudaMemcpyDeviceToDevice, st)) != cudaSuccess)
    return r;
  if (n > 0 && flags_out &&
      (r = cudaMemcpyAsync(flags_out, w.flags, n, cudaMemcpyDeviceToDevice, st)) != cudaSuccess)
    return r;
  return cudaGetLastError();
}

}  // namespace voc
}  // namespace ynb
