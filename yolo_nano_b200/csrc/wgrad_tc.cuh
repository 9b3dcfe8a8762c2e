// Weight gradient of the pointwise conv on tcgen05 tensor cores, fp32 parity mode (3xTF32):
//   dW[n][k] = sum_m dY[m][n] * X[m][k],   db[n] = sum_m dY[m][n]          (config 5, SURVEY §8 row a14)
// As an MMA:  D[128 x KPAD] += A[128 x 8] * B[KPAD x 8]^T with the PIXELS as the contraction dimension:
// A = dY^T (rows n), B = X^T (rows k).  Both activations are stored pixel-major ([m][channel]), i.e. the
// contraction index is the SLOW one, so the operands cannot be fetched by TMA into the K-major layout
// the MMA wants.  The threads have to touch every element anyway for the hi/lo split of the 3xTF32
// scheme, so the 8 producer warps do both at once: 16-byte loads (a lane = four channels of four consecutive
// pixels, a warp instruction = one whole 512-byte row), round-to-nearest split x = hi + lo, and a TRANSPOSING 16-byte store per plane
// into the 128-byte-swizzled K-major tiles (conflict-free: row = channel, chunk = pixel group ^ row % 8).
// Row K of the B tile is all ones, so column K of the accumulator is the bias gradient for free.
//
//   warps 0-7  producers (global -> split -> swizzled smem, mbarrier `full`), then the epilogue
//              (TMEM -> registers -> partial[chunk][N][K], main + correction accumulators added)
//   warp  8    one thread issues tcgen05.mma kind::tf32: per 8-pixel sub-step  main += A_hi*B_hi,
//              corr += A_lo*B_hi, corr += A_hi*B_lo; tcgen05.commit releases the stage (`empty`)
// One CTA per SM owns a contiguous range of pixels; the partials are summed in fixed order by
// reduce_partials_kernel (deterministic).  Every mbarrier wait is bounded (ptx::mbar_wait).
#pragma once
#include "common.cuh"
#include "ptx_sm100.cuh"

namespace ynb {

constexpr int kWgThreads = 288;
constexpr int kWgStepPix = 32;
constexpr uint32_t kWgABytes = 128 * 128;          // one A plane: 128 rows (n) x 32 floats of pixels

struct WgradParams {
  const float* dout; int do_ld, do_off;
  const float* in;   int in_ld, in_off;
  float* partial;                                  // [chunks][n tiles][128 rows][KPAD] in ACCUMULATOR order (permuted)
  long long M; int K, N;
  int stages;
  int H, W, dy, dx;                                // H > 0: tap (dy, dx) of a 3x3 conv (pad 1, stride 1): X row = pixel shifted by the
                                                   // tap, zero outside the image (the conv's padding); H = 0: pointwise
  int raw_slots;                                   // KPAD = 128: thread-private cp.async staging slots (0 = register path)
  long long steps_per_chunk;
  int* err;
};

__device__ __forceinline__ void split_tf32(float x, float& hi, float& lo) {
  hi = __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u);
  const float r = x - hi;                          // exact
  lo = __uint_as_float((__float_as_uint(r) + 0x1000u) & 0xffffe000u);
}

template <int KPAD>
__global__ void __launch_bounds__(kWgThreads, 1) pw_wgrad_tc_kernel(const WgradParams p) {
  extern __shared__ __align__(1024) uint8_t wg_smem_raw[];
  uint8_t* smem = wg_smem_raw + ((1024u - (ptx::smem_u32(wg_smem_raw) & 1023u)) & 1023u);
  __shared__ __align__(8) uint64_t full_bar[4], empty_bar[4], done_bar;
  __shared__ uint32_t tmem_ptr;
  constexpr uint32_t kBBytes = KPAD * 128;
  constexpr uint32_t kStageBytes = 2 * kWgABytes + 2 * kBBytes;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n0 = blockIdx.y * 128;
  const long long total_steps = (p.M + kWgStepPix - 1) / kWgStepPix;
  const long long s0 = (long long)blockIdx.x * p.steps_per_chunk;
  const long long s1 = s0 + p.steps_per_chunk < total_steps ? s0 + p.steps_per_chunk : total_steps;
  const int nsteps = s1 > s0 ? (int)(s1 - s0) : 0;
  const int stages = p.stages;

  if (threadIdx.x == 0) {
    for (int i = 0; i < 4; ++i) { ptx::mbar_init(&full_bar[i], 8); ptx::mbar_init(&empty_bar[i], 1); }
    ptx::mbar_init(&done_bar, 1);
    ptx::fence_barrier_init();
  }
  if (warp == 8) { ptx::tmem_alloc(&tmem_ptr, 512); ptx::tmem_relinquish(); }
  ptx::tc_fence_before_sync();
  __syncthreads();
  ptx::tc_fence_after_sync();
  const uint32_t tmem = tmem_ptr;

  if (warp < 8) {
    // ---------------- producers ----------------
    // Warp w owns pixels 4w .. 4w+3 of the step (= 16-byte chunk w of every tile row); a lane owns one
    // channel of a group of 32: four 128-byte coalesced row loads give it four consecutive pixels of its
    // channel = ONE 16-byte store per plane into row (32 i + lane), chunk (w ^ row % 8): conflict-free.
    const uint32_t in_row = (uint32_t)lane * 128u + ((uint32_t)(warp ^ (lane & 7)) << 4);
    // 16-byte loads: a lane reads channels 4*lane .. 4*lane+3 of four consecutive pixels (a warp = one whole
    // 512-byte row of 128 channels per instruction).  Channel 4*lane + c lives in tile row 32*c + lane (any
    // fixed permutation of the rows works - the epilogue undoes it), which keeps the stores conflict-free.
    // source pixel of X for output pixel m (3x3 tap: shifted, invalid outside the image)
    auto xsrc = [&](long long m, bool& ok) -> long long {
      ok = m < p.M;
      if (p.H > 0 && ok) {
        const int mi = (int)m;
        const int x = mi % p.W, y = (mi / p.W) % p.H;
        ok = (unsigned)(y + p.dy) < (unsigned)p.H && (unsigned)(x + p.dx) < (unsigned)p.W;
        return m + p.dy * p.W + p.dx;
      }
      return m;
    };
    auto load = [&](int t, float (&av)[16], float (&bv)[KPAD / 8]) {
      const long long m = (s0 + t) * kWgStepPix + 4 * warp;
      const float* drow = p.dout + m * p.do_ld + p.do_off + n0 + 4 * lane;
      const float* xrow = p.in + m * p.in_ld + p.in_off + 4 * lane;
      const bool aok = n0 + 4 * lane < p.N;                   // N, K are multiples of 4 on this path
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (aok && m + j < p.M) v = *reinterpret_cast<const float4*>(drow + (long long)j * p.do_ld);
        av[j] = v.x; av[4 + j] = v.y; av[8 + j] = v.z; av[12 + j] = v.w;
      }
#pragma unroll
      for (int g = 0; g < KPAD / 128; ++g) {
        const int k = 128 * g + 4 * lane;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (m + j < p.M) {
            bool xok;
            const long long xs = xsrc(m + j, xok);
            if (k < p.K) { if (xok) v = *reinterpret_cast<const float4*>(p.in + xs * p.in_ld + p.in_off + 4 * lane + 128 * g); }
            else if (k == p.K) v.x = 1.0f;                    // the ones row: accumulator column K = bias gradient
          }
          bv[16 * g + j] = v.x; bv[16 * g + 4 + j] = v.y; bv[16 * g + 8 + j] = v.z; bv[16 * g + 12 + j] = v.w;
        }
      }
    };
    auto store = [&](int t, const float (&av)[16], const float (&bv)[KPAD / 8]) {
      const int s = t % stages;
      if (t >= stages) ptx::mbar_wait(&empty_bar[s], ((t / stages) - 1) & 1, p.err, 1);
      uint8_t* st = smem + (size_t)s * kStageBytes;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float4 hi, lo;
        split_tf32(av[4 * i + 0], hi.x, lo.x); split_tf32(av[4 * i + 1], hi.y, lo.y);
        split_tf32(av[4 * i + 2], hi.z, lo.z); split_tf32(av[4 * i + 3], hi.w, lo.w);
        const uint32_t off = (uint32_t)i * 4096u + in_row;
        *reinterpret_cast<float4*>(st + off) = hi;
        *reinterpret_cast<float4*>(st + kWgABytes + off) = lo;
      }
#pragma unroll
      for (int i = 0; i < KPAD / 32; ++i) {
        float4 hi, lo;
        split_tf32(bv[4 * i + 0], hi.x, lo.x); split_tf32(bv[4 * i + 1], hi.y, lo.y);
        split_tf32(bv[4 * i + 2], hi.z, lo.z); split_tf32(bv[4 * i + 3], hi.w, lo.w);
        const uint32_t off = (uint32_t)i * 4096u + in_row;
        *reinterpret_cast<float4*>(st + 2 * kWgABytes + off) = hi;
        *reinterpret_cast<float4*>(st + 2 * kWgABytes + kBBytes + off) = lo;
      }
    };
    // fence.proxy.async compiles to MEMBAR.ALL.CTA + FENCE.VIEW.ASYNC: the membar DRAINS every outstanding
    // global load of the thread, so loads cannot be kept in flight across it.  Hence the loop works on PAIRS of
    // steps: both steps' loads are issued together (one DRAM latency per pair), both tiles are stored, ONE
    // fence publishes both stages.
    auto publish = [&](int t) {
      if (lane == 0) ptx::mbar_arrive(&full_bar[t % stages]);
    };
    if (KPAD == 128 && p.raw_slots > 0) {
      // Deep prefetch that survives the fence: the raw 16-byte pieces of the next steps travel global ->
      // shared with cp.async into THREAD-PRIVATE slots behind the operand stages (a thread reads back only
      // what it copied itself, so cp.async.wait_group is the only synchronisation).  cp.async copies are not
      // "outstanding loads" of the thread, so the membar of the proxy fence does not wait for them:
      // raw_slots - 1 whole steps stay in flight per thread.
      const int R = p.raw_slots;
      float4* rawbase = reinterpret_cast<float4*>(smem + (size_t)stages * kStageBytes);   // [R][8][256] float4
      auto issue = [&](int t) {
        if (t < nsteps) {
          const long long m = (s0 + t) * kWgStepPix + 4 * warp;
          float4* slot = rawbase + (size_t)(t % R) * 8 * 256 + threadIdx.x;
          const float* drow = p.dout + m * p.do_ld + p.do_off + n0 + 4 * lane;
          const float* xrow = p.in + m * p.in_ld + p.in_off + 4 * lane;
          const bool aok = n0 + 4 * lane < p.N, bok = 4 * lane < p.K;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const bool rok = m + j < p.M;
            ptx::cp_async_16(slot + j * 256, (rok && aok) ? (const void*)(drow + (long long)j * p.do_ld) : (const void*)p.dout,
                             (rok && aok) ? 16u : 0u);
            bool xok;
            const long long xs = xsrc(m + j, xok);
            ptx::cp_async_16(slot + (4 + j) * 256,
                             (xok && bok) ? (const void*)(p.in + xs * p.in_ld + p.in_off + 4 * lane) : (const void*)p.in,
                             (xok && bok) ? 16u : 0u);
          }
        }
        ptx::cp_async_commit();
      };
      for (int t = 0; t < R; ++t) issue(t);
      float av[16], bv[16];
#pragma unroll 1
      for (int t = 0; t < nsteps; ++t) {
        // groups committed so far: R + t; step t's group is complete when at most R - 1 are pending
        if (R == 3) asm volatile("cp.async.wait_group 2;" ::: "memory");
        else if (R == 2) asm volatile("cp.async.wait_group 1;" ::: "memory");
        else asm volatile("cp.async.wait_group 0;" ::: "memory");
        const float4* slot = rawbase + (size_t)(t % R) * 8 * 256 + threadIdx.x;
        const long long m = (s0 + t) * kWgStepPix + 4 * warp;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4 a = slot[j * 256];
          float4 b = slot[(4 + j) * 256];
          if (4 * lane == p.K && m + j < p.M) b.x = 1.0f;      // the ones row (bias gradient)
          av[j] = a.x; av[4 + j] = a.y; av[8 + j] = a.z; av[12 + j] = a.w;
          bv[j] = b.x; bv[4 + j] = b.y; bv[8 + j] = b.z; bv[12 + j] = b.w;
        }
        store(t, av, reinterpret_cast<const float (&)[KPAD / 8]>(bv));
        ptx::fence_proxy_async_smem();
        __syncwarp();
        publish(t);
        issue(t + R);                                          // refills the slot just consumed
      }
      asm volatile("cp.async.wait_group 0;" ::: "memory");
    } else {
    float av[2][16], bv[2][KPAD / 8];
    const int pair = stages >= 3 ? 2 : 1;          // with 2 stages a pair would serialise producers and MMA
#pragma unroll 1
    for (int t = 0; t < nsteps; t += pair) {
      const bool two = pair == 2 && t + 1 < nsteps;
      load(t, av[0], bv[0]);
      if (two) load(t + 1, av[1], bv[1]);
      store(t, av[0], bv[0]);
      if (two) store(t + 1, av[1], bv[1]);
      ptx::fence_proxy_async_smem();
      __syncwarp();
      publish(t);
      if (two) publish(t + 1);
    }
    }
    // ---------------- epilogue ----------------
    // The accumulator tile goes out as it sits in tensor memory (row = TMEM lane, 64 contiguous bytes per
    // lane and iteration: whole sectors); the row / column permutation of the producers and the padding are
    // undone ONCE by wgrad_reduce_kernel when it writes dW / db.
    const int lane_base = 32 * (warp & 3), half = warp >> 2;
    float* pt = p.partial + (((long long)blockIdx.x * gridDim.y + blockIdx.y) * 128 + lane_base + lane) * KPAD;
    if (nsteps > 0) {
      ptx::mbar_wait(&done_bar, 0, p.err, 2);
      ptx::tc_fence_after_sync();
    }
#pragma unroll 1
    for (int c0 = half * (KPAD / 2); c0 < (half + 1) * (KPAD / 2); c0 += 16) {
      uint32_t r1[16], r2[16];
      if (nsteps > 0) {
        ptx::tmem_ld_32x16(tmem + ((uint32_t)lane_base << 16) + (uint32_t)c0, r1);
        ptx::tmem_ld_32x16(tmem + ((uint32_t)lane_base << 16) + (uint32_t)(KPAD + c0), r2);
        ptx::tmem_ld_wait();
      } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) { r1[j] = 0u; r2[j] = 0u; }
      }
#pragma unroll
      for (int j = 0; j < 16; j += 4)
        *reinterpret_cast<float4*>(pt + c0 + j) =
            make_float4(__uint_as_float(r1[j]) + __uint_as_float(r2[j]), __uint_as_float(r1[j + 1]) + __uint_as_float(r2[j + 1]),
                        __uint_as_float(r1[j + 2]) + __uint_as_float(r2[j + 2]), __uint_as_float(r1[j + 3]) + __uint_as_float(r2[j + 3]));
    }
  } else {
    if (ptx::elect_one()) {   // elect.sync (not lane == 0): operands stay in uniform registers, MMAs issue back to back
    // ---------------- MMA issuer ----------------
    const uint32_t idesc = ptx::make_idesc(2, 128, KPAD);
    const uint32_t idesc2 = ptx::make_idesc(2, 128, KPAD == 128 ? 256 : KPAD);
    for (int t = 0; t < nsteps; ++t) {
      const int s = t % stages;
      ptx::mbar_wait(&full_bar[s], (t / stages) & 1, p.err, 3);
      ptx::tc_fence_after_sync();
      const uint32_t a_hi = ptx::smem_u32(smem + (size_t)s * kStageBytes), a_lo = a_hi + kWgABytes;
      const uint32_t b_hi = a_hi + 2 * kWgABytes, b_lo = b_hi + kBBytes;
#pragma unroll
      for (int sub = 0; sub < 4; ++sub) {
        const uint32_t ko = sub * 32;
        const uint32_t acc = (t | sub) != 0;
        if (KPAD == 128) {
          // [B_hi; B_lo] are adjacent in shared memory and [main | corr] adjacent in tensor memory: A_hi x both
          // is ONE instruction of N = 256 (an MMA costs the same for any N <= 256) - 2 instead of 3 per sub-step
          ptx::mma_tf32_ss(tmem, ptx::make_sw128_kmajor_desc(a_hi + ko), ptx::make_sw128_kmajor_desc(b_hi + ko), idesc2, acc);
          ptx::mma_tf32_ss(tmem + KPAD, ptx::make_sw128_kmajor_desc(a_lo + ko), ptx::make_sw128_kmajor_desc(b_hi + ko), idesc, 1u);
        } else {
          ptx::mma_tf32_ss(tmem, ptx::make_sw128_kmajor_desc(a_hi + ko), ptx::make_sw128_kmajor_desc(b_hi + ko), idesc, acc);
          ptx::mma_tf32_ss(tmem + KPAD, ptx::make_sw128_kmajor_desc(a_lo + ko), ptx::make_sw128_kmajor_desc(b_hi + ko), idesc, acc);
          ptx::mma_tf32_ss(tmem + KPAD, ptx::make_sw128_kmajor_desc(a_hi + ko), ptx::make_sw128_kmajor_desc(b_lo + ko), idesc, 1u);
        }
      }
      ptx::mma_commit(&empty_bar[s]);
    }
    if (nsteps > 0) ptx::mma_commit(&done_bar);
    }
    __syncwarp();
  }
  ptx::tc_fence_before_sync();
  __syncthreads();
  if (warp == 8) {
    ptx::tc_fence_after_sync();
    ptx::tmem_dealloc(tmem, 512);
  }
}

// Second stage: fixed-order sum over the chunks in accumulator order (coalesced), then ONE permuted write:
// tile row 32*c + l = output channel 4*l + c; column 128*g + 32*c + l = input channel 128*g + 4*l + c;
// column K = bias gradient.
// A block = 64 consecutive accumulator elements (16 threads x 16 bytes) x 32 chunk slices: every thread keeps
// chunks / 32 independent 16-byte loads in flight (the partials were just written: L2 reads).  Summation order per
// element: slice y adds chunks y, y + 32, ... ascending, then the slices 0..31 ascending — fixed, run-to-run identical.
constexpr int kWgRedElems = 64;
__global__ void __launch_bounds__(512) wgrad_reduce_kernel(const float* __restrict__ partial, int chunks, int ntiles,
                                                           int kpad, int N, int K, float* __restrict__ dw,
                                                           float* __restrict__ db) {
  __shared__ float4 sh[32][17];
  const long long elems = (long long)ntiles * 128 * kpad;          // multiple of 64
  const long long e = (long long)blockIdx.x * kWgRedElems + 4 * threadIdx.x;
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  if (e < elems)
    for (int j = threadIdx.y; j < chunks; j += 32) {
      const float4 v = *reinterpret_cast<const float4*>(partial + (long long)j * elems + e);
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
  sh[threadIdx.y][threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.y < 4 && e < elems) {          // 64 threads finish one element each: (x, component y)
    const int comp = threadIdx.y;
    float t = 0.0f;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const float4 v = sh[j][threadIdx.x];
      t += comp == 0 ? v.x : (comp == 1 ? v.y : (comp == 2 ? v.z : v.w));
    }
    const long long ee = e + comp;
    const int col = (int)(ee % kpad);
    const long long row = ee / kpad;
    const int r = (int)(row % 128), tile = (int)(row / 128);
    const int n = tile * 128 + 4 * (r & 31) + (r >> 5);
    const int k = (col & ~127) + 4 * (col & 31) + ((col >> 5) & 3);
    if (n < N) {
      if (k < K) dw[(long long)n * K + k] = t;
      else if (k == K) db[n] = t;
    }
  }
}
inline void launch_wgrad_reduce(const float* partial, int chunks, int ntiles, int kpad, int N, int K, float* dw, float* db,
                                cudaStream_t st) {
  const long long elems = (long long)ntiles * 128 * kpad;
  wgrad_reduce_kernel<<<(unsigned)((elems + kWgRedElems - 1) / kWgRedElems), dim3(16, 32), 0, st>>>(partial, chunks, ntiles, kpad,
                                                                                                  N, K, dw, db);
}

inline int wgrad_tc_kpad(int K) { return K + 1 <= 128 ? 128 : (K + 1 <= 256 ? 256 : 0); }
inline int wgrad_tc_chunks(long long M, int N) {
  const int ntile = (N + 127) / 128;
  long long chunks = kNumSMs / ntile;
  const long long total_steps = (M + kWgStepPix - 1) / kWgStepPix;
  if (chunks > total_steps) chunks = total_steps;
  return (int)(chunks < 1 ? 1 : chunks);
}

inline long long wgrad_tc_partial_floats(long long M, int K, int N) {
  return (long long)wgrad_tc_chunks(M, N) * ((N + 127) / 128) * 128 * wgrad_tc_kpad(K);
}

inline cudaError_t launch_pw_wgrad_tc(WgradParams p, int chunks, cudaStream_t st) {
  const int kpad = wgrad_tc_kpad(p.K);
  const long long total_steps = (p.M + kWgStepPix - 1) / kWgStepPix;
  p.steps_per_chunk = (total_steps + chunks - 1) / chunks;
  const size_t stage = 2 * kWgABytes + 2 * (size_t)kpad * 128;
  p.stages = 2;                                   // 2 operand stages (64 KB each at kpad 128)
  p.raw_slots = kpad == 128 ? 3 : 0;              // + 3 x 32 KB raw slots at kpad 128
  const size_t smem = stage * p.stages + (size_t)p.raw_slots * 32768 + 1024;
  dim3 grid(chunks, (p.N + 127) / 128);
  cudaError_t e;
  if (kpad == 128) {
    e = cudaFuncSetAttribute(pw_wgrad_tc_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    pw_wgrad_tc_kernel<128><<<grid, kWgThreads, smem, st>>>(p);
  } else {
    e = cudaFuncSetAttribute(pw_wgrad_tc_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    pw_wgrad_tc_kernel<256><<<grid, kWgThreads, smem, st>>>(p);
  }
  YNB_COUNT_LAUNCH();
  return cudaGetLastError();
}

}  // namespace ynb
