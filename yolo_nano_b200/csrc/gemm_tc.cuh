// tcgen05 tensor-core contraction for the dense convs of the path (pointwise 1x1 and the
// 3x3 "smooth" convs as implicit GEMM), fed by TMA, accumulating in TMEM.
//
//   D[m, n] = act(bias[n] + sum_k A[m, k] * W[n, k])       m: NHWC pixels, k: channels
//
// Tile: 128 pixel rows x Npad (<= 256) output channels; K consumed in chunks of 32 floats
// (one 128-byte swizzle row).  A persistent CTA walks its tiles; five roles:
//   warps 0-3   epilogue group 0  TMEM -> regs -> bias/act -> swizzled smem box -> TMA store /
//   warps 4-7   epilogue group 1  coalesced (interleaved) row stores; group g owns TMEM stage g
//   warps 8-11  splitters         fp32 parity mode only: A -> (A_hi, A_lo) in smem
//   warp 12     TMA producer      A chunk (+ W chunk when W is streamed) -> smem stage
//   warp 13     MMA issuer        tcgen05.mma kind::tf32, one elected lane; owns TMEM alloc
//
// fp32 parity mode (YNB_GEMM_TC_3XTF32): a*b ~= a_hi*b_hi + a_hi*b_lo + a_lo*b_hi with
// x_hi = RN_tf32(x), x_lo = RN_tf32(x - x_hi): three MMAs per K step.  Measured on B200
// (tools/gpu_accum_probe.py, profiles/):
//   * a truncating split (x & 0xffffe000) leaves a -2.7e-7 relative bias and 4.4e-7 rms
//     (the dropped a_lo*b_lo term is then one-signed); round-to-nearest makes the split
//     unbiased with 9.5e-8 rms — hence RN;
//   * the tensor core TRUNCATES when it adds into the accumulator: bias ~ -0.4 ulp per
//     accumulation step (K=464: -2.9e-6 on one-signed sums, FFMA: 1e-9).  The small correction
//     products must therefore not be added into the large sum: they get their OWN accumulator and
//     the epilogue adds main + correction in fp32 (one merged accumulator doubles the end-to-end
//     error; spreading the main products over several accumulators buys nothing measurable).
//     With main and correction adjacent in TMEM and W_hi / W_lo adjacent in smem,
//     a_hi x [b_hi; b_lo] is ONE MMA of N = 2*Npad (`stack_b`): two MMAs per K step.
// W_hi / W_lo are split once at weight-pack time; A is split in shared memory by the
// splitter warps, position-wise on the swizzled bytes (no layout knowledge needed) — or once
// by the kernel that produces it (`presplit`, 3x3 convs: two TMA boxes per step, no splitters).
//
// Epilogue variants: plain (TMA bulk tensor store of the swizzled box), pass-through
// interleave (stride-1 ShuffleNet unit tail: out[2i] = x1[i], out[2i+1] = conv[i]), slot-mapped /
// spatial-tile stores, and the fused detection decode (kDecC = 80 | 20).  The CTA's last tile is
// drained by both epilogue groups, half of the columns each.
//
// 3x3 mode: the nine taps are nine TMA boxes of the same 4-D tensor map shifted by
// (dx-1, dy-1); out-of-bounds elements are zero-filled by TMA = the conv's zero padding.
#pragma once
#include <cuda.h>

#include <cstring>

#include "common.cuh"
#include "ptx_sm100.cuh"

namespace ynb {

constexpr int kTcThreads = 512;
constexpr int kTcSplitWarp0 = 8, kTcProducerWarp = 12, kTcMmaWarp = 13;   // warps 0-7: two epilogue groups
constexpr int kTcProducers = 3;                                            // producer roles: warps 12, 14, 15
constexpr int kTcBM = 128;
constexpr int kTcBK = 32;                       // floats per K chunk = 128 bytes
constexpr int kTcAStageBytes = kTcBM * 128;     // 16 KB
constexpr int kTcMaxStages = 8;
constexpr int kTcSmemBudget = 232448;                   // 227 KB opt-in maximum (layout totals include the alignment slack)

struct TcGemmParams {
  int num_steps;          // K chunks per tile (pointwise: ceil(K/32); 3x3: 9 * C/32)
  int chunks_per_tap;     // 3x3: C/32; pointwise: num_steps
  int is3x3;
  int mode;               // YNB_GEMM_TC_3XTF32 | YNB_GEMM_TC_TF32 | YNB_GEMM_TC_BF16
  int bf16_in;            // A and W are bf16 (K chunk = 64 elements = the same 128 bytes): kind::f16, one pass
  int out_bf16;           // the output tensor is bf16 (fp32 accumulators, bias and activation; rounded on store)
  int num_stages;
  int w_resident;
  int64_t M;              // pointwise: rows
  int64_t num_tiles;
  int H, W, TH, TW, tiles_x, tiles_y;   // 3x3 spatial tiling
  int N, Npad;
  int nacc;               // accumulators per stage: 2 (main + correction) in parity mode unless merged, else 1
  int merge_corr;         // parity mode, shallow K: corrections go into the single main accumulator (nacc = 1)
  int ksub;               // pointwise: valid 8-float K sub-steps = ceil(K / 8) (sub-steps made only of zero padding are
                          // not issued: K = 116 needs 15 of 16, K = 232 29 of 32, K = 24 3 of 4); 0 = all
  int presplit;           // parity mode, 3x3: A arrives as two planes (hi, lo) written by the producer kernel —
                          // two TMA boxes per step, no splitter pass (tmAlo)
  int a2_step;            // pointwise, > 0: K steps [a2_step, num_steps) read a SECOND activation tensor (tmAlo) — the
                          // two branches of a stride-2 ShuffleNetV2 unit concatenated along K against block-diagonal,
                          // row-interleaved weights: torch.cat + channel_shuffle as one plain GEMM output
  int stack_b;            // parity mode, 2*Npad <= 256: a_hi x [b_hi; b_lo] as ONE MMA of N = 2*Npad
                          // into [main | corr] (the planes are adjacent in smem and in TMEM): 2 MMAs per
                          // K-step instead of 3, a_hi and b_hi are fetched once less
  int acc_stages;         // TMEM accumulator stages (2 = epilogue overlaps the next tile's MMAs)
  uint32_t tmem_cols;     // power of two >= acc_stages * nacc * Npad
  uint32_t a_box_bytes;   // bytes one A TMA box delivers
  // epilogue
  float* out;
  int out_ld, out_off, out_step;
  const float* bias;
  int act;
  // Stride-1 ShuffleNetV2 unit: this GEMM is branch2's last conv; `pass` points at the
  // pass-through half x1 (same pixels, `N` channels).  The epilogue then writes whole
  // interleaved rows out[2i] = x1[i], out[2i+1] = branch2[i]  — torch.cat +
  // channel_shuffle (backbone/shufflenetv2.py:70-76, 14-28) as one coalesced store.
  const float* pass;
  int pass_ld;
  int tma_store;          // plain pointwise outputs leave through TMA bulk tensor stores (tmOut)
  // Fused detection decode (head_det_*.4): instead of writing the raw [M, A(1+C+4)] map, the
  // epilogue thread that owns a pixel row turns it into boxes / scores / classes
  // (models/yolo_nano.py:303-330, 120-156, 362-367, 253-256) — the largest activation of the
  // network never reaches HBM.
  struct Decode {
    float* boxes;        // [B, Ntot, 4]
    float* scores;       // [B, Ntot]
    int32_t* cls;        // [B, Ntot]
    int G, HW;           // grid side, cells per image
    float stride, input_size;
    float aw[3], ah[3];
    int64_t Ntot, level_off;
  } dec;
  int* err_flag;
  // debug timeline (tools/gpu_tc_trace.py): CTA 0 appends {role, tile, step, clock64}
  long long* trace;
  int trace_cap;
};

// roles: 1 producer-issued, 2 split-done, 3 mma-issued, 4 epilogue-start, 5 epilogue-end, 6 tile accumulators ready
// Non-intrusive: every (role, local tile, step) has its own slot — plain stores, no atomics, no
// round trip in the traced thread (an atomic counter costs ~1000 cycles per event and paces the
// very loops being observed).  Slots: ((role * 64 + local_tile % 64) * 32 + step % 32) * 4.
#define YNB_TRACE(role, a, b)                                                                        \
  do {                                                                                               \
    if (p.trace != nullptr && blockIdx.x == 0) {                                                     \
      const int _lt = (int)(((long long)(a) - (long long)blockIdx.x) / (long long)gridDim.x) & 63;   \
      long long* _e = p.trace + 1 + (long long)((((role) * 64 + _lt) * 32) + ((int)(b) & 31)) * 4;   \
      _e[0] = (role); _e[1] = (a); _e[2] = (b); _e[3] = clock64();                                   \
    }                                                                                                \
  } while (0)

struct TcSmemLayout {
  uint32_t stage_bytes;    // A | A_lo | (W_hi | W_lo when streamed)
  uint32_t w_chunk_bytes;  // Npad * 128
  uint32_t w_res_off;      // offset of the resident W region
  uint32_t bias_off;
  uint32_t stg_off;        // per-epilogue-warp transpose staging (interleaved stores)
  uint32_t bar_off;
  uint32_t total;
};
constexpr int kTcStgBytes = 8 * 4096;                            // 8 epilogue warps x one swizzled [32 rows x 128 B] box

__host__ __device__ inline TcSmemLayout tc_smem_layout(int Npad, int num_steps, int num_stages, bool w_resident,
                                                       bool split) {
  TcSmemLayout L;
  L.w_chunk_bytes = (uint32_t)Npad * 128;
  uint32_t a_bytes = kTcAStageBytes * (split ? 2 : 1);
  uint32_t w_bytes = w_resident ? 0 : L.w_chunk_bytes * (split ? 2 : 1);
  L.stage_bytes = a_bytes + w_bytes;                      // all multiples of 1024
  L.w_res_off = L.stage_bytes * num_stages;
  uint32_t w_res = w_resident ? L.w_chunk_bytes * (split ? 2 : 1) * num_steps : 0;
  L.bias_off = L.w_res_off + w_res;
  L.stg_off = L.bias_off + 1024;                          // bias: up to 256 floats (keeps 1024-B alignment)
  L.bar_off = L.stg_off + kTcStgBytes;
  L.total = L.bar_off + 256 + 1024;                       // barriers + slack for 1024-B alignment
  return L;
}

// round-to-nearest (ties away) to TF32 on the raw bits; exact for values already in TF32
__host__ __device__ __forceinline__ uint32_t rn_tf32_bits(uint32_t u) { return (u + 0x1000u) & 0xffffe000u; }

template <bool kPass, int kDecC>
__global__ void __launch_bounds__(kTcThreads, 1)
tc_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmAlo,
               const __grid_constant__ CUtensorMap tmWhi, const __grid_constant__ CUtensorMap tmWlo,
               const __grid_constant__ CUtensorMap tmOut, const TcGemmParams p) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  // 1024-byte alignment (128-byte swizzle atoms) by OFFSET arithmetic on the __shared__ array,
  // so that every access below stays in the shared address space (LDS / STS, not generic)
  uint8_t* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);

  const bool split = p.mode == YNB_GEMM_TC_3XTF32;
  const int kchunk = p.bf16_in ? 64 : kTcBK;       // elements per K chunk (128 bytes)
  // TMA boxes per K step: A (hi) [, A_lo when pre-split] [, W_hi [, W_lo] when W is streamed].  Issuing a
  // box costs the issuing thread ~600 cycles whatever its size (tools/tma_probe.cu), and that cost
  // overlaps across warps (1 issuer 27 B/clk/SM, 2: 54, 4: 104) — so the boxes of a step are spread over
  // up to three producer warps instead of being issued one after the other by one.
  const int box_alo = p.presplit ? 1 : -1;
  const int box_whi = p.w_resident ? -1 : 1 + (p.presplit ? 1 : 0);
  const int box_wlo = (p.w_resident || !split) ? -1 : box_whi + 1;
  const int nboxes = 1 + (box_alo >= 0) + (box_whi >= 0) + (box_wlo >= 0);
  const int nprod = nboxes < kTcProducers ? nboxes : kTcProducers;
  const TcSmemLayout lay = tc_smem_layout(p.Npad, p.num_steps, p.num_stages, p.w_resident != 0, split);
  const uint32_t w_chunk_bytes = lay.w_chunk_bytes;
  const uint32_t a_bytes = kTcAStageBytes * (split ? 2 : 1);
  const uint32_t stage_bytes = lay.stage_bytes;
  const uint32_t w_res_bytes = lay.bias_off - lay.w_res_off;
  float* s_bias = reinterpret_cast<float*>(smem + lay.bias_off);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + lay.bar_off);
  uint64_t* full = bars;                         // [kTcMaxStages]  TMA landed
  uint64_t* ready = bars + kTcMaxStages;         // [kTcMaxStages]  A split done (parity mode)
  uint64_t* empty = bars + 2 * kTcMaxStages;     // [kTcMaxStages]  MMAs retired, stage reusable
  uint64_t* tmem_full = bars + 3 * kTcMaxStages;       // [2]
  uint64_t* tmem_empty = bars + 3 * kTcMaxStages + 2;  // [2]
  uint64_t* w_full = bars + 3 * kTcMaxStages + 4;      // [1]
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 3 * kTcMaxStages + 5);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  pdl_trigger();

  if (warp == kTcProducerWarp && lane == 0) {
    ptx::prefetch_tmap(&tmA);
    if (p.presplit || p.a2_step > 0) ptx::prefetch_tmap(&tmAlo);
    ptx::prefetch_tmap(&tmWhi);
    if (split) ptx::prefetch_tmap(&tmWlo);
    if (p.tma_store) ptx::prefetch_tmap(&tmOut);
    for (int s = 0; s < p.num_stages; ++s) {
      ptx::mbar_init(&full[s], nprod);   // one arrive.expect_tx per producer role
      ptx::mbar_init(&ready[s], 4);      // one arrival per splitter warp
      ptx::mbar_init(&empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(&tmem_full[a], 1);
      ptx::mbar_init(&tmem_empty[a], 4); // one arrival per warp of the epilogue group that owns the stage
    }
    ptx::mbar_init(w_full, 1);
    ptx::fence_barrier_init();
  }
  if (warp == kTcMmaWarp) {
    ptx::tmem_alloc(tmem_ptr, p.tmem_cols);
    ptx::tmem_relinquish();
  }
  if (warp < 4) {    // stage the bias once (no global latency inside the tile loop)
    for (int i = threadIdx.x; i < p.Npad; i += 128) s_bias[i] = i < p.N ? __ldg(p.bias + i) : 0.0f;
  }
  ptx::tc_fence_before_sync();
  __syncthreads();
  ptx::tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_ptr;

  auto stage_a = [&](int s) { return smem + (size_t)s * stage_bytes; };
  auto stage_alo = [&](int s) { return smem + (size_t)s * stage_bytes + kTcAStageBytes; };
  auto w_hi_ptr = [&](int s, int step) {
    return p.w_resident ? smem + lay.w_res_off + (size_t)step * w_chunk_bytes * (split ? 2 : 1)
                        : smem + (size_t)s * stage_bytes + a_bytes;
  };
  auto w_lo_ptr = [&](int s, int step) { return w_hi_ptr(s, step) + w_chunk_bytes; };

  const int acc_cols = p.Npad * p.nacc;   // TMEM columns per accumulator stage
  const uint32_t step_tx = p.a_box_bytes * (p.presplit ? 2 : 1) + (p.w_resident ? 0 : w_chunk_bytes * (split ? 2 : 1));
  const bool splitters_on = split && !p.presplit;

  // Weights do not depend on the previous kernel: the resident W planes are requested before
  // the programmatic-dependency wait, i.e. while the predecessor is still draining.
  if (warp == kTcProducerWarp && p.w_resident && ptx::elect_one()) {
    ptx::mbar_arrive_expect_tx(w_full, w_res_bytes);
    for (int st = 0; st < p.num_steps; ++st) {
      ptx::tma_load_2d(w_hi_ptr(0, st), &tmWhi, w_full, st * kchunk, 0);
      if (split) ptx::tma_load_2d(w_lo_ptr(0, st), &tmWlo, w_full, st * kchunk, 0);
    }
  }
  pdl_wait();

  const int prole = warp == kTcProducerWarp ? 0 : (warp == 14 ? 1 : (warp == 15 ? 2 : -1));
  if (prole >= 0) {
    // ================= TMA producers (role r issues the boxes j with j % nprod == r) =================
    // elect.sync in a warp-uniform branch (not `lane == 0`): the compiler then knows a single thread runs the
    // loop and keeps descriptors / coordinates in UNIFORM registers — no R2UR + ELECT waterfall loop around
    // every UTMALDG / UTCHMMA (measured, tools/mma_probe2.cu: 142 -> 67 cycles per issued MMA).
    if (prole < nprod && ptx::elect_one()) {
      const bool do_a = 0 % nprod == prole;
      const bool do_alo = box_alo >= 0 && box_alo % nprod == prole;
      const bool do_whi = box_whi >= 0 && box_whi % nprod == prole;
      const bool do_wlo = box_wlo >= 0 && box_wlo % nprod == prole;
      const uint32_t my_tx = (do_a ? p.a_box_bytes : 0u) + (do_alo ? p.a_box_bytes : 0u) +
                             (do_whi ? w_chunk_bytes : 0u) + (do_wlo ? w_chunk_bytes : 0u);
      int s = 0;
      uint32_t ph = 0;
      bool ok = true;
      for (int64_t tile = blockIdx.x; tile < p.num_tiles && ok; tile += gridDim.x) {
        int b = 0, y0 = 0, x0 = 0;
        if (p.is3x3) {
          int per_img = p.tiles_x * p.tiles_y;
          b = (int)(tile / per_img);
          int r = (int)(tile - (int64_t)b * per_img);
          y0 = (r / p.tiles_x) * p.TH;
          x0 = (r % p.tiles_x) * p.TW;
        }
        for (int st = 0; st < p.num_steps; ++st) {
          ok = ptx::mbar_wait(&empty[s], ph ^ 1, p.err_flag, 1);
          if (!ok) break;
          ptx::mbar_arrive_expect_tx(&full[s], my_tx);
          if (p.is3x3) {
            int tap = st / p.chunks_per_tap, kc = st - tap * p.chunks_per_tap;
            int dy = tap / 3, dx = tap - dy * 3;
            if (do_a) ptx::tma_load_4d(stage_a(s), &tmA, &full[s], kc * kchunk, x0 + dx - 1, y0 + dy - 1, b);
            if (do_alo) ptx::tma_load_4d(stage_alo(s), &tmAlo, &full[s], kc * kchunk, x0 + dx - 1, y0 + dy - 1, b);
          } else {
            if (do_a) {
              const bool second = p.a2_step > 0 && st >= p.a2_step;
              ptx::tma_load_2d(stage_a(s), second ? &tmAlo : &tmA, &full[s], (second ? st - p.a2_step : st) * kchunk,
                               (int)(tile * kTcBM));
            }
          }
          if (do_whi) ptx::tma_load_2d(w_hi_ptr(s, st), &tmWhi, &full[s], st * kchunk, 0);
          if (do_wlo) ptx::tma_load_2d(w_lo_ptr(s, st), &tmWlo, &full[s], st * kchunk, 0);
          if (prole == 0) YNB_TRACE(1, tile, st);
          if (++s == p.num_stages) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == kTcMmaWarp) {
    // ================= MMA issuer =================
    if (ptx::elect_one()) {
      const uint32_t idesc = ptx::make_idesc(2 /*tf32*/, kTcBM, p.Npad);
      const uint32_t idesc2 = ptx::make_idesc(2, kTcBM, 2 * p.Npad);
      const uint32_t idesc_bf = ptx::make_idesc(1 /*bf16*/, kTcBM, p.Npad);
      int s = 0;
      uint32_t ph = 0;
      int acc = 0;
      uint32_t acc_ph = 0;
      bool ok = true;
      if (p.w_resident) ok = ptx::mbar_wait(w_full, 0, p.err_flag, 2);
      for (int64_t tile = blockIdx.x; tile < p.num_tiles && ok; tile += gridDim.x) {
        ok = ptx::mbar_wait(&tmem_empty[acc], acc_ph ^ 1, p.err_flag, 3);
        if (!ok) break;
        ptx::tc_fence_after_sync();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * acc_cols);
        // correction accumulator (the main one itself when merged: its first MMA initialises it)
        const uint32_t c_tmem = p.merge_corr ? d_tmem : d_tmem + (uint32_t)p.Npad;
        int t = 0;                                                       // K-step counter of the tile
        for (int st = 0; st < p.num_steps; ++st) {
          ok = ptx::mbar_wait(splitters_on ? &ready[s] : &full[s], ph, p.err_flag, 4);
          if (!ok) break;
          ptx::tc_fence_after_sync();
          const uint32_t a_hi = ptx::smem_u32(stage_a(s));
          const uint32_t a_lo = ptx::smem_u32(stage_alo(s));
          const uint32_t b_hi = ptx::smem_u32(w_hi_ptr(s, st));
          const uint32_t b_lo = ptx::smem_u32(w_lo_ptr(s, st));
          const int nk = p.ksub > 0 ? min(kTcBK / 8, p.ksub - st * (kTcBK / 8)) : kTcBK / 8;
          // one code path per arithmetic mode (the issue loop is latency-critical: no per-MMA mode tests)
          if (p.bf16_in) {
#pragma unroll
            for (int k = 0; k < kTcBK / 8; ++k, ++t) {
              if (k >= nk) break;
              ptx::mma_bf16_ss(d_tmem, ptx::make_sw128_kmajor_desc(a_hi + k * 32), ptx::make_sw128_kmajor_desc(b_hi + k * 32),
                               idesc_bf, t != 0);
            }
          } else if (p.stack_b) {
#pragma unroll
            for (int k = 0; k < kTcBK / 8; ++k, ++t) {
              if (k >= nk) break;
              const uint64_t db = ptx::make_sw128_kmajor_desc(b_hi + k * 32);
              // [main | corr] (+)= a_hi x [b_hi; b_lo]   then   corr += a_lo x b_hi
              ptx::mma_tf32_ss(d_tmem, ptx::make_sw128_kmajor_desc(a_hi + k * 32), db, idesc2, t != 0);
              ptx::mma_tf32_ss(c_tmem, ptx::make_sw128_kmajor_desc(a_lo + k * 32), db, idesc, 1);
            }
          } else {
#pragma unroll
            for (int k = 0; k < kTcBK / 8; ++k, ++t) {
              if (k >= nk) break;
              const uint32_t ko = k * 32;   // 8 tf32 = 32 bytes inside the 128-byte swizzled row
              const uint64_t da = ptx::make_sw128_kmajor_desc(a_hi + ko);
              const uint64_t db = ptx::make_sw128_kmajor_desc(b_hi + ko);
              if (split) {
                ptx::mma_tf32_ss(c_tmem, ptx::make_sw128_kmajor_desc(a_lo + ko), db, idesc, t != 0);
                ptx::mma_tf32_ss(c_tmem, da, ptx::make_sw128_kmajor_desc(b_lo + ko), idesc, 1);
              }
              ptx::mma_tf32_ss(d_tmem, da, db, idesc, (split && p.merge_corr) ? 1 : (t != 0));
            }
          }
          YNB_TRACE(3, tile, st);
          ptx::mma_commit(&empty[s]);                       // frees the smem stage when the MMAs retire
          if (st == p.num_steps - 1) ptx::mma_commit(&tmem_full[acc]);
          if (++s == p.num_stages) { s = 0; ph ^= 1; }
        }
        if (++acc == p.acc_stages) { acc = 0; acc_ph ^= 1; }
      }
    }
  } else if (warp >= kTcSplitWarp0 && warp < kTcSplitWarp0 + 4) {
    // ================= splitters (fp32 parity mode) =================
    if (splitters_on) {
      const int t = threadIdx.x - kTcSplitWarp0 * 32;  // 0..127
      int s = 0;
      uint32_t ph = 0;
      bool ok = true;
      for (int64_t tile = blockIdx.x; tile < p.num_tiles && ok; tile += gridDim.x) {
        for (int st = 0; st < p.num_steps; ++st) {
          ok = ptx::mbar_wait(&full[s], ph, p.err_flag, 5);
          if (!ok) break;
          uint4* a = reinterpret_cast<uint4*>(stage_a(s));
          uint4* lo = reinterpret_cast<uint4*>(stage_alo(s));
#pragma unroll
          for (int i = 0; i < kTcAStageBytes / 16 / 128; ++i) {
            const uint4 v = a[t + i * 128];
            uint4 h, l;
            h.x = rn_tf32_bits(v.x); h.y = rn_tf32_bits(v.y); h.z = rn_tf32_bits(v.z); h.w = rn_tf32_bits(v.w);
            l.x = rn_tf32_bits(__float_as_uint(__uint_as_float(v.x) - __uint_as_float(h.x)));
            l.y = rn_tf32_bits(__float_as_uint(__uint_as_float(v.y) - __uint_as_float(h.y)));
            l.z = rn_tf32_bits(__float_as_uint(__uint_as_float(v.z) - __uint_as_float(h.z)));
            l.w = rn_tf32_bits(__float_as_uint(__uint_as_float(v.w) - __uint_as_float(h.w)));
            a[t + i * 128] = h;
            lo[t + i * 128] = l;
          }
          ptx::fence_proxy_async_smem();     // generic-proxy writes -> visible to the tensor core
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&ready[s]);
          if (t == 0) YNB_TRACE(2, tile, st);
          if (++s == p.num_stages) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp < 8) {
    // ================= epilogue: two groups of four warps =================
    // Group g owns accumulator stage g and the tiles with (local index % 2) == g, so the
    // TMEM drain + stores of tile i overlap those of tile i+1 (and the MMAs of tile i+2).
    // With a single accumulator stage group 1 stays idle.
    const int group = warp >> 2;
    const int q = warp & 3;                         // TMEM lane quarter this warp may read
    const int row = q * 32 + lane;                  // tile row owned by this thread
    const bool vec = p.out_step == 1;
    const float slope = p.act == YNB_ACT_RELU ? 0.0f : (p.act == YNB_ACT_LEAKY ? 0.1f : 1.0f);
    uint8_t* sbox = smem + lay.stg_off + warp * 4096;          // this warp's [32 rows x 128 B] swizzled box
    const int sw = lane & 7;                                    // swizzle phase of this thread's row
    // The LAST tile of this CTA is drained by BOTH groups, half of the columns each: nothing is left to
    // overlap with, so the kernel's tail (one epilogue: 7 k cycles plain, 18 k interleaved) halves.
    // Not for the decode epilogue (a thread needs all columns of its row).
    const int nloc = (int64_t)blockIdx.x < p.num_tiles
                         ? (int)((p.num_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x) : 0;   // tiles of this CTA
    const bool share_last = kDecC == 0;
    const int col_split = min(p.Npad, ((p.Npad / 2 + 31) / 32) * 32);      // group 0: [0, split), group 1: [split, Npad)
    bool ok = true;
    for (int lt = 0; lt < nloc && ok; ++lt) {
      const int64_t tile = blockIdx.x + (int64_t)lt * gridDim.x;
      const int acc = p.acc_stages == 2 ? (lt & 1) : 0;
      const bool shared = share_last && lt == nloc - 1 && col_split < p.Npad;
      if (!shared && group != acc) {                            // owner group only
        // With ONE accumulator stage group 1 owns nothing: it still observes every phase of the barrier,
        // so that its parity wait for the shared last tile cannot match an older phase.  (With two stages
        // the non-owner has just drained tile lt-1, whose completion implies tile lt-2's — in-order commits.)
        if (p.acc_stages == 1 && share_last) ok = ptx::mbar_wait(&tmem_full[0], (uint32_t)(lt & 1), p.err_flag, 7);
        continue;
      }
      const int col_begin = shared && group == 1 ? col_split : 0;
      const int col_end = shared && group == 0 ? col_split : p.Npad;
      const uint32_t acc_ph = (uint32_t)((lt / p.acc_stages) & 1);
      // row -> output pixel
      int64_t m;
      bool valid;
      if (p.is3x3) {
        int per_img = p.tiles_x * p.tiles_y;
        int b = (int)(tile / per_img);
        int r = (int)(tile - (int64_t)b * per_img);
        int y = (r / p.tiles_x) * p.TH + row / p.TW;
        int x = (r % p.tiles_x) * p.TW + row % p.TW;
        valid = row < p.TH * p.TW && y < p.H && x < p.W;
        m = ((int64_t)b * p.H + y) * p.W + x;
      } else {
        m = tile * kTcBM + row;
        valid = m < p.M;
      }
      // Pass-through prefetch (interleave mode): the x1 values this warp will store do not
      // depend on the MMAs, so the loads of the first 32-channel block are issued BEFORE
      // waiting for the accumulator, and each half (16 rows) is re-armed for the next block
      // right after it has been stored.
      const int64_t m_base = tile * kTcBM + q * 32;            // first row of this warp (pointwise)
      float xa[16], xb[16];
      // one 64-bit address per call, 32-bit row offsets after that (the math was 22 % of the kernel's
      // instructions when every row recomputed m * ld in 64 bits)
      const int rows_left = (int)min((int64_t)32, p.M - m_base);   // valid rows of this warp's 32 (<= 0: none)
      auto fetch_x1 = [&](int c0, int r0, float (&x)[16]) {
        const int i = c0 + lane;
        const bool col_ok = kPass && i < p.N;
        const float* src = p.pass + (m_base + r0) * (int64_t)p.pass_ld + i;
        const int nr = col_ok ? rows_left - r0 : 0;
#pragma unroll
        for (int r = 0; r < 16; ++r) x[r] = r < nr ? __ldg(src + r * p.pass_ld) : 0.0f;
      };
      if (kPass) {
        fetch_x1(col_begin, 0, xa);
        fetch_x1(col_begin, 16, xb);
      }
      if (lane == 0 && q == 0) YNB_TRACE(4, tile, group);
      ok = ptx::mbar_wait(&tmem_full[acc], acc_ph, p.err_flag, 6);
      if (!ok) break;
      ptx::tc_fence_after_sync();
      if (lane == 0 && q == 0) YNB_TRACE(6, tile, group);
      const uint32_t t_base = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * acc_cols);
      if constexpr (kDecC > 0) {
        // ================= fused decode epilogue (one pixel = one thread) =================
        // Round 2: the fully unrolled column walk was ~15 k instructions (250 KB of SASS) and ran at ~70 cycles per
        // column — instruction-cache bound.  Now ROLLED loops over 16-column blocks per anchor (class logits of
        // anchor a are columns [A + a*C, A + (a+1)*C): a tcgen05.ld may start at any column), two passes as before
        // (max + first arg-max, then the softmax denominator) — the same values in the same order as
        // decode_level_kernel, bit for bit.
        constexpr int A = 3, C = kDecC, CB = (C + 15) / 16;
        auto ld16 = [&](int c0, float (&v)[16]) {          // 16 raw columns: accumulator sum(s), no bias yet
          uint32_t r[16];
          ptx::tmem_ld_32x16(t_base + c0, r);
          if (p.nacc == 2) {
            uint32_t r2[16];
            ptx::tmem_ld_32x16(t_base + (uint32_t)p.Npad + c0, r2);
            ptx::tmem_ld_wait();
#pragma unroll
            for (int jj = 0; jj < 16; ++jj) r[jj] = __float_as_uint(__uint_as_float(r[jj]) + __uint_as_float(r2[jj]));
          }
          ptx::tmem_ld_wait();
#pragma unroll
          for (int jj = 0; jj < 16; ++jj) v[jj] = __uint_as_float(r[jj]);
        };
        float objl[A], mx[A], sum[A], tb[4 * A];
        int am[A];
        {   // objectness logits: columns [0, A); box logits: columns [A + A*C, A + A*C + 4A)
          float v[16];
          ld16(0, v);
#pragma unroll
          for (int a = 0; a < A; ++a) objl[a] = v[a] + s_bias[a];
          // (the 16-column read must stay inside this accumulator stage: start at most at Npad - 16)
          constexpr int NPADC = (A * (1 + C + 4) + 15) / 16 * 16;
          constexpr int B0 = (A + A * C) < (NPADC - 16) ? (A + A * C) : (NPADC - 16);
          constexpr int BOFF = A + A * C - B0;
          ld16(B0, v);
#pragma unroll
          for (int k = 0; k < 4 * A; ++k) tb[k] = v[BOFF + k] + s_bias[A + A * C + k];
        }
#pragma unroll
        for (int a = 0; a < A; ++a) {
          const int cbase = A + a * C;
          float m = -INFINITY;
          int arg = 0;
#pragma unroll 1
          for (int blk = 0; blk < CB; ++blk) {              // pass 1: class max + first arg-max
            float v[16];
            ld16(cbase + blk * 16, v);
            const float* bb = s_bias + cbase + blk * 16;
#pragma unroll
            for (int jj = 0; jj < 16; ++jj) {
              const int c = blk * 16 + jj;
              const float x = v[jj] + bb[jj];
              if ((C % 16 == 0 || c < C) && x > m) { m = x; arg = c; }
            }
          }
          float sm = 0.0f;
#pragma unroll 1
          for (int blk = 0; blk < CB; ++blk) {              // pass 2: softmax denominator (TMEM re-read: cheaper than 3*C registers)
            float v[16];
            ld16(cbase + blk * 16, v);
            const float* bb = s_bias + cbase + blk * 16;
#pragma unroll
            for (int jj = 0; jj < 16; ++jj) {
              const int c = blk * 16 + jj;
              if (C % 16 == 0 || c < C) sm += softmax_exp((v[jj] + bb[jj]) - m);
            }
          }
          mx[a] = m; am[a] = arg; sum[a] = sm;
        }
        (void)mx;
        {   // all TMEM reads of this tile are done: hand the stage back
          ptx::tc_fence_before_sync();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&tmem_empty[acc]);
        }
        if (valid) {
          const int b = (int)(m / p.dec.HW);
          const int pix = (int)(m - (int64_t)b * p.dec.HW);
          const int gy = pix / p.dec.G, gx = pix - gy * p.dec.G;
          const int64_t o0 = (int64_t)b * p.dec.Ntot + p.dec.level_off + (int64_t)pix * A;
#pragma unroll
          for (int a = 0; a < A; ++a) {
            const float obj = 1.0f / (1.0f + expf(-objl[a]));
            const float score = class_score(sum[a], obj);
            const float tx = tb[4 * a], ty = tb[4 * a + 1], tw = tb[4 * a + 2], th = tb[4 * a + 3];
            float cx = __fmul_rn(__fadd_rn(1.0f / (1.0f + expf(-tx)), (float)gx), p.dec.stride);
            float cy = __fmul_rn(__fadd_rn(1.0f / (1.0f + expf(-ty)), (float)gy), p.dec.stride);
            float w = __fmul_rn(expf(tw), p.dec.aw[a]);
            float h = __fmul_rn(expf(th), p.dec.ah[a]);
            float hw = __fmul_rn(w, 0.5f), hh = __fmul_rn(h, 0.5f);
            float x1 = __fdiv_rn(__fsub_rn(cx, hw), p.dec.input_size);
            float y1 = __fdiv_rn(__fsub_rn(cy, hh), p.dec.input_size);
            float x2 = __fdiv_rn(__fadd_rn(cx, hw), p.dec.input_size);
            float y2 = __fdiv_rn(__fadd_rn(cy, hh), p.dec.input_size);
            reinterpret_cast<float4*>(p.dec.boxes)[o0 + a] =
                make_float4(fminf(fmaxf(x1, 0.f), 1.f), fminf(fmaxf(y1, 0.f), 1.f), fminf(fmaxf(x2, 0.f), 1.f),
                            fminf(fmaxf(y2, 0.f), 1.f));
            p.dec.scores[o0 + a] = score;
            p.dec.cls[o0 + a] = am[a];
          }
        }
        if (lane == 0 && q == 0) YNB_TRACE(5, tile, group);
        continue;
      }
      // 16 columns: sum of the accumulators (main + correction) + bias, activation
      // (branch-free: act(x) = max(x, slope*x), slope 1 / 0 / 0.1 = identity / ReLU / LeakyReLU(0.1)),
      // written as chunks jc..jc+3 of this thread's swizzled 128-byte line
      // The previous TMA store of this warp must have finished READING the staging box before it is rewritten: waited
      // for after the accumulator loads of the box's first 16 columns, whose latency covers it.
      auto box_free = [&]() {
        if (p.tma_store) {
          if (ptx::elect_one()) ptx::bulk_wait_read<0>();
          __syncwarp();
        }
      };
      auto drain16 = [&](int c0, int jc) {
        uint32_t r[16];
        ptx::tmem_ld_32x16(t_base + c0, r);
        if (p.nacc == 2) {            // main + correction: both loads, one wait
          uint32_t r2[16];
          ptx::tmem_ld_32x16(t_base + (uint32_t)p.Npad + c0, r2);
          ptx::tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 16; ++j) r[j] = __float_as_uint(__uint_as_float(r[j]) + __uint_as_float(r2[j]));
        } else {
          ptx::tmem_ld_wait();
        }
        if (jc == 0) box_free();
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4 b4 = *reinterpret_cast<const float4*>(s_bias + c0 + 4 * j);
          float x0 = __uint_as_float(r[4 * j]) + b4.x, x1 = __uint_as_float(r[4 * j + 1]) + b4.y;
          float x2 = __uint_as_float(r[4 * j + 2]) + b4.z, x3 = __uint_as_float(r[4 * j + 3]) + b4.w;
          *reinterpret_cast<float4*>(sbox + lane * 128 + (((jc + j) ^ sw) << 4)) =
              make_float4(fmaxf(x0, x0 * slope), fmaxf(x1, x1 * slope), fmaxf(x2, x2 * slope), fmaxf(x3, x3 * slope));
        }
      };
      // value (row r, column l of the block) back out of the swizzled box
      auto staged = [&](int r, int l) {
        return *reinterpret_cast<const float*>(sbox + r * 128 + ((((l >> 2) ^ (r & 7)) << 4) | ((l & 3) << 2)));
      };

      // bf16 output through TMA: this thread's 16 columns as 32 bytes of its dense 64-byte staging row
      auto drain16_bf16 = [&](int c0, int half) {
        uint32_t r[16];
        ptx::tmem_ld_32x16(t_base + c0, r);
        ptx::tmem_ld_wait();
        if (half == 0) box_free();
        uint32_t w[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float x0 = __uint_as_float(r[2 * j]) + s_bias[c0 + 2 * j], x1 = __uint_as_float(r[2 * j + 1]) + s_bias[c0 + 2 * j + 1];
          w[j] = pack_bf16x2(fmaxf(x0, x0 * slope), fmaxf(x1, x1 * slope));
        }
        uint4* dst = reinterpret_cast<uint4*>(sbox + lane * 64 + half * 32);
        dst[0] = make_uint4(w[0], w[1], w[2], w[3]);
        dst[1] = make_uint4(w[4], w[5], w[6], w[7]);
      };
      const bool bf16_box = p.out_bf16 && p.tma_store && !kPass;
      bf16* const out_bf = reinterpret_cast<bf16*>(p.out);

      for (int c0 = col_begin; c0 < col_end; c0 += 32) {
        if (bf16_box) {
          drain16_bf16(c0, 0);
          if (c0 + 16 < col_end) drain16_bf16(c0 + 16, 1);
        } else {
          drain16(c0, 0);
          if (c0 + 16 < col_end) drain16(c0 + 16, 4);
        }
        if (c0 + 32 >= col_end && !shared) {   // all TMEM reads of this tile are done: hand the stage back
          ptx::tc_fence_before_sync();          // (a shared tile is the CTA's last: nobody waits for the stage)
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&tmem_empty[acc]);
        }
        if (!kPass && p.tma_store) {
          // ---- plain pointwise output: the swizzled box leaves through one TMA store ----
          ptx::fence_proxy_async_smem();
          __syncwarp();
          if (ptx::elect_one()) {
            ptx::tma_store_2d(&tmOut, sbox, c0, (int)m_base);   // rows >= M / cols >= N4 are clipped
            ptx::bulk_commit();
          }
          continue;
        }
        __syncwarp();
        const int i = c0 + lane;                                // output channel of this lane
        const bool col_ok = i < p.N;
        if (kPass) {
          // out[2i] = x1[i] (pass-through), out[2i+1] = branch2[i]: 256-byte row segments
          const int nrow = col_ok ? (int)min((int64_t)32, p.M - m_base) : 0;   // rows this lane stores
          float* o = p.out + m_base * p.out_ld + 2 * (col_ok ? i : 0);
#pragma unroll
          for (int r = 0; r < 16; ++r, o += p.out_ld)
            if (r < nrow) *reinterpret_cast<float2*>(o) = make_float2(xa[r], staged(r, lane));
          if (c0 + 32 < col_end) fetch_x1(c0 + 32, 0, xa);
#pragma unroll
          for (int r = 16; r < 32; ++r, o += p.out_ld)
            if (r < nrow) *reinterpret_cast<float2*>(o) = make_float2(xb[r - 16], staged(r, lane));
          if (c0 + 32 < col_end) fetch_x1(c0 + 32, 16, xb);
        } else {
          const int col = p.out_off + (vec ? i : (col_ok ? i : 0) * p.out_step);
          if (!p.is3x3) {
            const int nrow = col_ok ? (int)min((int64_t)32, p.M - m_base) : 0;
            if (p.out_bf16) {
              bf16* o = out_bf + m_base * p.out_ld + col;
#pragma unroll 8
              for (int r = 0; r < 32; ++r, o += p.out_ld)
                if (r < nrow) *o = __float2bfloat16_rn(staged(r, lane));
            } else {
              float* o = p.out + m_base * p.out_ld + col;
#pragma unroll 8
              for (int r = 0; r < 32; ++r, o += p.out_ld)
                if (r < nrow) *o = staged(r, lane);
            }
          } else {
            // spatial tile: row -> pixel is not affine, take it from the lane that owns the row
            const int64_t off = valid ? m * p.out_ld : -1;
#pragma unroll 8
            for (int r = 0; r < 32; ++r) {
              const int64_t offr = __shfl_sync(0xffffffffu, off, r);
              if (col_ok && offr >= 0) {
                if (p.out_bf16) out_bf[offr + col] = __float2bfloat16_rn(staged(r, lane));
                else p.out[offr + col] = staged(r, lane);
              }
            }
          }
        }
        __syncwarp();
      }
      if (lane == 0 && q == 0) YNB_TRACE(5, tile, group);
    }
    __syncwarp();
    if (p.tma_store && ptx::elect_one()) ptx::bulk_wait<0>();   // all output boxes have landed
  }

  ptx::tc_fence_before_sync();
  __syncthreads();
  if (warp == kTcMmaWarp) {
    ptx::tc_fence_after_sync();
    ptx::tmem_dealloc(tmem_base, p.tmem_cols);
  }
}

// --------------------------------------------------------------------------------------
// host side
// --------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                    CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                    CUtensorMapFloatOOBfill);

inline PFN_encodeTiled get_encode_tiled() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_encodeTiled>(p);
  }
  return fn;
}

// rank-2 map over a K-major matrix (fp32, or bf16 with `bf16` set): dim0 = K (contiguous), dim1 = rows; boxes of
// 128 bytes of K (32 floats | 64 bf16) x box_rows.  Strides / extents in ELEMENTS.
inline bool make_tmap_2d(CUtensorMap* m, const void* base, uint64_t k, uint64_t rows, uint64_t row_stride_elems,
                         uint32_t box_rows, bool bf16 = false) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc) return false;
  const uint64_t es = bf16 ? 2 : 4;
  cuuint64_t dims[2] = {k, rows};
  cuuint64_t strides[1] = {row_stride_elems * es};
  cuuint32_t box[2] = {(cuuint32_t)(128 / es), box_rows};
  cuuint32_t estr[2] = {1, 1};
  return enc(m, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), dims,
             strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
             CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// rank-4 map over an NHWC activation [B][H][W][ld] exposing C channels: (c, x, y, b); boxes of 128 bytes of
// channels (32 floats | 64 bf16) x box_w x box_h pixels.
inline bool make_tmap_nhwc(CUtensorMap* m, const void* base, int C, int W, int H, int B, int ld, int box_w,
                           int box_h, bool bf16 = false, bool swizzle = true) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc) return false;
  const uint64_t es = bf16 ? 2 : 4;
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
  cuuint64_t strides[3] = {(cuuint64_t)ld * es, (cuuint64_t)ld * es * W, (cuuint64_t)ld * es * W * H};
  cuuint32_t box[4] = {(cuuint32_t)(128 / es), (cuuint32_t)box_w, (cuuint32_t)box_h, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  return enc(m, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<void*>(base), dims,
             strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             swizzle ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
             CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// rank-4 map over the NCHW fp32 network input [B][3][S][S] for the stem: boxes of
// [40 x 35 x 3 x 1] floats, no swizzle, zero fill outside the image (the conv's padding).  The start
// coordinate of the innermost dimension must keep the global address 16-byte aligned.
inline bool make_tmap_stem_input(CUtensorMap* m, const float* x, int S, int B) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc || (reinterpret_cast<uintptr_t>(x) & 15u) || (S & 3)) return false;
  cuuint64_t dims[4] = {(cuuint64_t)S, (cuuint64_t)S, 3, (cuuint64_t)B};
  cuuint64_t strides[3] = {(cuuint64_t)S * 4, (cuuint64_t)S * S * 4, (cuuint64_t)S * S * 12};
  cuuint32_t box[4] = {40, 35, 3, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  return enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(x), dims, strides, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// rank-2 STORE map over an output view [rows][ld] exposing `cols` channels (multiple of 4):
// boxes of 32 channels x 32 rows, 128-byte swizzle (matches the epilogue's staging layout).
// bf16: the staging box is [32 rows x 64 bytes] (32 bf16 columns), no swizzle.
inline bool make_tmap_out(CUtensorMap* m, void* base, uint64_t cols, uint64_t rows, uint64_t ld, bool bf16 = false) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc) return false;
  const uint64_t es = bf16 ? 2 : 4;
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {ld * es};
  cuuint32_t box[2] = {32, 32};
  cuuint32_t estr[2] = {1, 1};
  return enc(m, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, base, dims, strides, box,
             estr, CU_TENSOR_MAP_INTERLEAVE_NONE, bf16 ? CU_TENSOR_MAP_SWIZZLE_NONE : CU_TENSOR_MAP_SWIZZLE_128B,
             CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// Weights packed for the tensor-core path: [Npad][Kpad] fp32, Kpad multiple of 32, split
// into exact-tf32 hi and lo parts.
struct TcWeights {
  float* hi = nullptr;
  float* lo = nullptr;
  bf16* bw = nullptr;     // bf16 mode: ONE plane [Npad][Kpad], Kpad multiple of 64; tm_hi maps it, tm_lo unused
  int N = 0, Npad = 0, Kpad = 0;
  CUtensorMap tm_hi, tm_lo;
};

inline void split_tf32_host(float v, float* hi, float* lo) {
  uint32_t u;
  memcpy(&u, &v, 4);
  uint32_t h = rn_tf32_bits(u);
  float hf;
  memcpy(&hf, &h, 4);
  float l = v - hf;
  uint32_t lu;
  memcpy(&lu, &l, 4);
  lu = rn_tf32_bits(lu);
  memcpy(lo, &lu, 4);
  *hi = hf;
}

// A fully described launch (tensor maps are baked at plan time).
struct TcGemmLaunch {
  CUtensorMap tmA;
  CUtensorMap tmOut;      // valid when p.tma_store
  const TcWeights* w = nullptr;
  CUtensorMap tmAlo;      // lo plane of A (presplit) | second activation tensor (a2_step > 0)
  TcGemmParams p;
  uint32_t smem = 0;
  unsigned grid = 0;
  int dec_classes = 0;    // 80 | 20: fused decode epilogue (p.dec valid); 0: ordinary epilogue
};

// TMEM plan (512 columns).  Parity mode: one main accumulator plus one correction accumulator.
// Measured (B200, calibrated weights, 128^2 and 416^2): with the round-to-nearest split and the
// corrections in their own accumulator, ONE main accumulator gives the same end-to-end error as
// four round-robin ones (box error 0.024 vs 0.025 px, identical keep sets) — and it lets the hi/lo
// weight planes be stacked into one MMA and the 3x3 convs double-buffer their accumulators: 3x3
// convs 2x faster.  Two accumulator stages (epilogue of tile i overlaps the MMAs of tile i+1)
// whenever they fit.
inline void tc_plan_tmem(TcGemmParams& p, bool allow_merge = false) {
  const bool split = p.mode == YNB_GEMM_TC_3XTF32;
  // <= 16 K steps (48 accumulations): the one-sided truncation of a single accumulator stays
  // below 3e-6 relative — buys two accumulator stages for N = 256 (fused decode heads)
  p.merge_corr = (split && allow_merge && p.num_steps * (kTcBK / 8) <= 16 && 2 * p.Npad <= 512) ? 1 : 0;
  p.nacc = split && !p.merge_corr ? 2 : 1;
  p.acc_stages = 2 * p.nacc * p.Npad <= 512 ? 2 : 1;
  p.tmem_cols = 32;
  while ((int)p.tmem_cols < p.acc_stages * p.nacc * p.Npad) p.tmem_cols <<= 1;
  p.stack_b = (p.nacc == 2 && 2 * p.Npad <= 256 && (2 * p.Npad) % 16 == 0) ? 1 : 0;
}

// Picks stages / residency for the smem budget.  Returns false if nothing fits.
inline bool tc_plan_smem(TcGemmLaunch& L) {
  TcGemmParams& p = L.p;
  const bool split = p.mode == YNB_GEMM_TC_3XTF32;
  for (int resident = 1; resident >= 0; --resident) {
    for (int stages = kTcMaxStages; stages >= 2; --stages) {
      if (stages > p.num_steps * 4 && stages > 2) continue;
      TcSmemLayout lay = tc_smem_layout(p.Npad, p.num_steps, stages, resident != 0, split);
      if (lay.total <= (uint32_t)kTcSmemBudget && (resident == 0 || stages >= 3 || p.num_steps <= 2)) {
        p.num_stages = stages;
        p.w_resident = resident;
        L.smem = lay.total;
        return true;
      }
    }
  }
  return false;
}

inline cudaError_t launch_tc_gemm(const TcGemmLaunch& L, cudaStream_t st) {
  using KernelT = void (*)(CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, TcGemmParams);
  static const KernelT kernels[4] = {tc_gemm_kernel<false, 0>, tc_gemm_kernel<true, 0>, tc_gemm_kernel<false, 80>,
                                     tc_gemm_kernel<false, 20>};
  static bool attr_set = false;
  if (!attr_set) {
    for (KernelT k : kernels) {
      cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, kTcSmemBudget);
      if (e != cudaSuccess) return e;
    }
    attr_set = true;
  }
  const CUtensorMap& tmo = L.p.tma_store ? L.tmOut : L.tmA;   // unused unless tma_store
  KernelT kern = L.dec_classes == 80 ? kernels[2] : (L.dec_classes == 20 ? kernels[3] : kernels[L.p.pass != nullptr ? 1 : 0]);
  const CUtensorMap& tmalo = (L.p.presplit || L.p.a2_step > 0) ? L.tmAlo : L.tmA;   // unused otherwise
  cudaError_t r = launch_pdl(kern, dim3(L.grid), dim3(kTcThreads), (size_t)L.smem, st, L.tmA, tmalo, L.w->tm_hi,
                             L.w->tm_lo, tmo, L.p);
  YNB_COUNT_LAUNCH();
  return r;
}

// Spatial tile (TW x TH <= 128 pixels) for the 3x3 path that wastes the fewest MMA rows.
inline void tc_pick_tile(int H, int W, int* TH, int* TW) {
  double best = -1;
  for (int tw = 4; tw <= 64 && tw <= W + 3; ++tw) {
    int th = 128 / tw;
    if (th < 1) continue;
    if (th > H) th = H;
    double eff = (double)H * W / ((double)((W + tw - 1) / tw) * ((H + th - 1) / th) * 128.0);
    if (eff > best + 1e-9) { best = eff; *TH = th; *TW = tw; }
  }
}

}  // namespace ynb
