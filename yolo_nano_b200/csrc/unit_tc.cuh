// Fused depthwise 3x3 -> pointwise 1x1 unit tail on tcgen05 (one launch instead of two, the depthwise
// output never reaches HBM):
//
//   stride-1 ShuffleNetV2 unit (backbone/shufflenetv2.py:53-63, 70-76):
//       mid1 --dw3x3+BN--> (smem) --pw+BN+ReLU--> out[2i+1],  x1[i] -> out[2i]
//   detection-head pair (models/yolo_nano.py:50-58):
//       x --dw3x3+BN+Leaky--> (smem) --pw+BN+Leaky--> out
//
// The kernel boundary sits at the depthwise INPUT: that is where a halo exchange between tiles is needed
// anyway, and L2 serves it (a tile re-reads a 1-pixel ring of its neighbours' pixels).  One CTA per SM walks
// spatial tiles of TH x TW <= 128 output pixels (the 128 rows of one UMMA tile):
//
//   warp 16      TMA producer: the tile WITH ITS HALO, 32 channels at a time, as ONE 4-D box
//                [(TH+2) x (TW+2) pixels x 32 ch], 128-byte swizzle, out-of-image pixels zero-filled by the
//                copy engine (= the conv's padding), into a 2..4-deep "raw" ring (as deep as shared memory
//                allows: the bytes in flight per SM bound the HBM rate); L2 prefetch of the pass-through tile
//   warp 18      TMA producer for the weight chunks when W does not fit in shared memory (streamed)
//   warps 8-15   depthwise producers: 3x3 taps with packed FFMA2 from the raw tile (a thread = 1x4 output strip
//                x 4 channels, sliding window in registers), + bias (+ LeakyReLU), split into exact-tf32
//                hi / lo (fp32 parity mode) and stored as rows of the K-major, 128-byte-swizzled A operand
//   warp 17      tcgen05.mma issuer (kind::tf32; [main | corr] (+)= a_hi x [b_hi; b_lo], corr += a_lo x b_hi)
//   warps 0-7    two epilogue groups, one per TMEM accumulator stage: the thread that owns a tile row builds
//                its output row (interleaved with the pass-through half for ShuffleNet units) in a swizzled
//                staging box, the warp copies the box out 16 bytes per lane
//
// Storage type E = float (fp32 parity / tf32 modes: K chunks of 32 channels, A split into hi / lo planes) or
// bf16 (YNB_GEMM_TC_BF16: K chunks of 64 channels — the same 128 bytes per row —, kind::f16 MMAs, one plane);
// depthwise taps, bias, activations and accumulators are fp32 in both.
//
// Arithmetic is identical to the unfused pair (dwconv3x3_tma_kernel + tc_gemm_kernel): same FFMA2 tap order,
// same split, same MMAs — the fused and unfused paths agree bit for bit on the depthwise values and to the
// accumulation order on the GEMM.
#pragma once
#include "gemm_tc.cuh"

namespace ynb {

constexpr int kDpThreads = 640;
constexpr int kDpEpiWarps = 8;                    // warps 0-7: two epilogue groups (group g owns TMEM accumulator stage g)
constexpr int kDpDwWarp0 = 8, kDpDwWarps = 8;     // warps 8-15: depthwise producers, ONE task per thread and chunk
constexpr int kDpRawWarp = 16, kDpMmaWarp = 17, kDpWWarp = 18;
constexpr int kDpMaxAStages = 4, kDpMaxRawStages = 4;
constexpr int kDpStgBytes = kDpEpiWarps * 4096;   // one swizzled [32 rows x 128 B] box per epilogue warp

struct DwPwParams {
  int H, W, lgTW, tiles_x, tiles_y;   // tile = TW x TH output pixels, TW = 1 << lgTW in {16, 32}, TH = 128 / TW
  int64_t num_tiles;
  int C4;             // depthwise channels (= K of the pointwise conv), physical width of the input view
  int num_chunks;     // K chunks of 32 channels
  int ksub;           // valid 8-channel sub-steps = ceil(C / 8)
  int N, Npad;
  int mode;           // YNB_GEMM_TC_3XTF32 | YNB_GEMM_TC_TF32
  int w_resident, a_stages, raw_stages;
  int pass_blocks;    // 32-channel blocks of the pass-through half to prefetch into L2 per tile (0: none)
  int tma_out;        // every warp's staging box leaves through ONE TMA tensor store (tmOut)
  uint32_t tmem_cols;
  const float* dw_w;  // [9][C4] tap-major, BN folded
  const float* dw_b;  // [C4]
  int dw_act;
  float* out;
  int out_ld, out_off;
  const float* bias;
  int act;
  const float* pass;  // stride-1 unit: x1 (same pixels, N channels) -> out[2i]; conv -> out[2i+1]
  int pass_ld;
  int* err_flag;
  long long* trace;   // debug timeline (tools/gpu_dp_trace.py): CTA 0 stores clock64 at [role][local tile][chunk]
};

// roles: 0 raw issued, 1 raw landed (seen by dw warp 0), 2 A written, 3 MMAs issued, 4 accumulator ready (epilogue), 5 epilogue done
#define YNB_DP_TRACE(role, lt, kc)                                                              \
  do {                                                                                           \
    if (p.trace != nullptr && blockIdx.x == 0 && (lt) < 16)                                      \
      p.trace[((role) * 16 + (lt)) * 8 + ((kc) & 7)] = clock64();                               \
  } while (0)

struct DpSmemLayout {
  uint32_t raw_stride, a_off, a_stride, w_chunk_bytes, w_res_off, dww_off, bias_off, stg_off, bar_off, total;
};

__host__ __device__ inline DpSmemLayout dp_smem_layout(int Npad, int num_chunks, int lgTW, int a_stages, int raw_stages,
                                                       bool w_resident, bool split, int chunk_ch = 32) {
  DpSmemLayout L;
  const int TW = 1 << lgTW, TH = kTcBM >> lgTW;
  L.w_chunk_bytes = (uint32_t)Npad * 128;
  L.raw_stride = ((uint32_t)((TW + 2) * (TH + 2) * 128) + 1023u) & ~1023u;
  L.a_off = L.raw_stride * raw_stages;
  L.a_stride = kTcAStageBytes * (split ? 2 : 1) + (w_resident ? 0 : L.w_chunk_bytes * (split ? 2 : 1));
  L.w_res_off = L.a_off + L.a_stride * a_stages;
  const uint32_t w_res = w_resident ? L.w_chunk_bytes * (split ? 2 : 1) * num_chunks : 0;
  L.dww_off = L.w_res_off + w_res;
  L.bias_off = L.dww_off + (((uint32_t)(10 * num_chunks * chunk_ch * 4) + 1023u) & ~1023u);   // 9 taps + bias
  L.stg_off = L.bias_off + 1024;
  L.bar_off = L.stg_off + kDpStgBytes;
  L.total = L.bar_off + 256 + 1024;
  return L;
}

// fp32 -> tf32, round to nearest (ties away): same bits as rn_tf32_bits() for finite values, one instruction
__device__ __forceinline__ float cvt_rna_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}

template <bool kPass, typename E>
__global__ void __launch_bounds__(kDpThreads, 1)
dwpw_tc_kernel(const __grid_constant__ CUtensorMap tmIn, const __grid_constant__ CUtensorMap tmWhi,
               const __grid_constant__ CUtensorMap tmWlo, const __grid_constant__ CUtensorMap tmPass,
               const __grid_constant__ CUtensorMap tmOut, const DwPwParams p) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);

  constexpr bool kBf16 = sizeof(E) == 2;
  constexpr int CH = 128 / (int)sizeof(E);          // channels per K chunk (one 128-byte swizzle row): 32 | 64
  constexpr int CGS = CH / 4;                       // 4-channel groups per chunk: 8 | 16
  const bool split = !kBf16 && p.mode == YNB_GEMM_TC_3XTF32;
  const DpSmemLayout lay = dp_smem_layout(p.Npad, p.num_chunks, p.lgTW, p.a_stages, p.raw_stages, p.w_resident != 0, split, CH);
  const uint32_t w_chunk_bytes = lay.w_chunk_bytes;
  const int KC = p.num_chunks * CH;
  const int TW = 1 << p.lgTW, TH = kTcBM >> p.lgTW;
  float* s_dww = reinterpret_cast<float*>(smem + lay.dww_off);     // [10][KC]: taps 0..8, row 9 = bias
  float* s_bias = reinterpret_cast<float*>(smem + lay.bias_off);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + lay.bar_off);
  uint64_t* raw_full = bars;            // [4]  TMA landed the halo tile chunk
  uint64_t* raw_empty = bars + 4;       // [4]  depthwise producers are done with it
  uint64_t* a_ready = bars + 8;         // [4]  A operand (hi, lo) of the stage written
  uint64_t* a_empty = bars + 12;        // [4]  MMAs of the stage retired
  uint64_t* w_full = bars + 16;         // [4]  streamed W chunk landed (resident: [0] once)
  uint64_t* tmem_full = bars + 20;      // [2]
  uint64_t* tmem_empty = bars + 22;     // [2]
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 24);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  pdl_trigger();

  if (warp == kDpRawWarp && lane == 0) {
    ptx::prefetch_tmap(&tmIn);
    ptx::prefetch_tmap(&tmWhi);
    if (split) ptx::prefetch_tmap(&tmWlo);
    if (p.pass_blocks) ptx::prefetch_tmap(&tmPass);
    if (p.tma_out) ptx::prefetch_tmap(&tmOut);
    for (int s = 0; s < kDpMaxRawStages; ++s) {
      ptx::mbar_init(&raw_full[s], 1);
      ptx::mbar_init(&raw_empty[s], kBf16 ? kDpDwWarps : kDpDwWarps / 2);   // the warps of ONE producer group
    }
    for (int s = 0; s < kDpMaxAStages; ++s) {
      ptx::mbar_init(&a_ready[s], kBf16 ? kDpDwWarps : kDpDwWarps / 2);
      ptx::mbar_init(&a_empty[s], 1);
      ptx::mbar_init(&w_full[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(&tmem_full[a], 1);
      ptx::mbar_init(&tmem_empty[a], 4);
    }
    ptx::fence_barrier_init();
  }
  if (warp == kDpMmaWarp) {
    ptx::tmem_alloc(tmem_ptr, p.tmem_cols);
    ptx::tmem_relinquish();
  }
  // depthwise taps + bias and the pointwise bias, staged once (weights do not depend on the previous kernel)
  for (int i = threadIdx.x; i < 10 * KC; i += kDpThreads) {
    const int tap = i / KC, c = i - tap * KC;
    float v = 0.0f;
    if (c < p.C4) v = tap < 9 ? __ldg(p.dw_w + tap * p.C4 + c) : __ldg(p.dw_b + c);
    s_dww[i] = v;
  }
  for (int i = threadIdx.x; i < p.Npad; i += kDpThreads) s_bias[i] = i < p.N ? __ldg(p.bias + i) : 0.0f;
  ptx::tc_fence_before_sync();
  __syncthreads();
  ptx::tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_ptr;

  const int nacc = split ? 2 : 1;
  const int acc_cols = p.Npad * nacc;
  const int per_img = p.tiles_x * p.tiles_y;
  auto a_stage = [&](int s) { return smem + lay.a_off + (size_t)s * lay.a_stride; };
  auto w_hi_ptr = [&](int s, int kc) {
    return p.w_resident ? smem + lay.w_res_off + (size_t)kc * w_chunk_bytes * (split ? 2 : 1)
                        : a_stage(s) + kTcAStageBytes * (split ? 2 : 1);
  };

  if (warp == kDpRawWarp && p.w_resident && ptx::elect_one()) {
    ptx::mbar_arrive_expect_tx(&w_full[0], w_chunk_bytes * (split ? 2 : 1) * p.num_chunks);
    for (int kc = 0; kc < p.num_chunks; ++kc) {
      ptx::tma_load_2d(w_hi_ptr(0, kc), &tmWhi, &w_full[0], kc * CH, 0);
      if (split) ptx::tma_load_2d(w_hi_ptr(0, kc) + w_chunk_bytes, &tmWlo, &w_full[0], kc * CH, 0);
    }
  }
  pdl_wait();

  if (warp == kDpRawWarp) {
    // ================= TMA producer: halo tiles =================
    if (ptx::elect_one()) {
      const uint32_t raw_bytes = (uint32_t)((TW + 2) * (TH + 2) * 128);
      int r = 0;
      uint32_t ph = 0;
      bool ok = true;
      for (int64_t tile = blockIdx.x; tile < p.num_tiles && ok; tile += gridDim.x) {
        const int b = (int)(tile / per_img);
        const int rr = (int)(tile - (int64_t)b * per_img);
        const int y0 = (rr / p.tiles_x) * TH, x0 = (rr % p.tiles_x) * TW;
        // the pass-through half of this tile is read by the epilogue a few microseconds from now: pull it into L2
#pragma unroll 1
        for (int cb = 0; cb < p.pass_blocks; ++cb) ptx::tma_prefetch_4d(&tmPass, cb * CH, x0, y0, b);
        for (int kc = 0; kc < p.num_chunks; ++kc) {
          ok = ptx::mbar_wait(&raw_empty[r], ph ^ 1, p.err_flag, 1);
          if (!ok) break;
          ptx::mbar_arrive_expect_tx(&raw_full[r], raw_bytes);
          ptx::tma_load_4d(smem + (size_t)r * lay.raw_stride, &tmIn, &raw_full[r], kc * CH, x0 - 1, y0 - 1, b);
          YNB_DP_TRACE(0, (int)((tile - blockIdx.x) / gridDim.x), kc);
          if (++r == p.raw_stages) { r = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == kDpWWarp) {
    // ================= TMA producer: streamed weight chunks =================
    if (!p.w_resident && ptx::elect_one()) {
      int s = 0;
      uint32_t ph = 0;
      bool ok = true;
      for (int64_t tile = blockIdx.x; tile < p.num_tiles && ok; tile += gridDim.x) {
        for (int kc = 0; kc < p.num_chunks; ++kc) {
          ok = ptx::mbar_wait(&a_empty[s], ph ^ 1, p.err_flag, 2);
          if (!ok) break;
          ptx::mbar_arrive_expect_tx(&w_full[s], w_chunk_bytes * (split ? 2 : 1));
          ptx::tma_load_2d(w_hi_ptr(s, kc), &tmWhi, &w_full[s], kc * CH, 0);
          if (split) ptx::tma_load_2d(w_hi_ptr(s, kc) + w_chunk_bytes, &tmWlo, &w_full[s], kc * CH, 0);
          if (++s == p.a_stages) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == kDpMmaWarp) {
    // ================= MMA issuer =================
    if (ptx::elect_one()) {
      const uint32_t idesc = ptx::make_idesc(kBf16 ? 1 : 2 /*bf16 | tf32*/, kTcBM, p.Npad);
      const uint32_t idesc2 = ptx::make_idesc(2, kTcBM, 2 * p.Npad);
      const bool stack_b = split && 2 * p.Npad <= 256;
      int s = 0, acc = 0;
      uint32_t ph = 0, acc_ph = 0;
      bool ok = true;
      if (p.w_resident) ok = ptx::mbar_wait(&w_full[0], 0, p.err_flag, 3);
      for (int64_t tile = blockIdx.x; tile < p.num_tiles && ok; tile += gridDim.x) {
        ok = ptx::mbar_wait(&tmem_empty[acc], acc_ph ^ 1, p.err_flag, 4);
        if (!ok) break;
        ptx::tc_fence_after_sync();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * acc_cols);
        const uint32_t c_tmem = d_tmem + (uint32_t)p.Npad;
        for (int kc = 0; kc < p.num_chunks; ++kc) {
          ok = ptx::mbar_wait(&a_ready[s], ph, p.err_flag, 5);
          if (ok && !p.w_resident) ok = ptx::mbar_wait(&w_full[s], ph, p.err_flag, 6);
          if (!ok) break;
          ptx::tc_fence_after_sync();
          const uint32_t a_hi = ptx::smem_u32(a_stage(s));
          const uint32_t a_lo = a_hi + kTcAStageBytes;
          const uint32_t b_hi = ptx::smem_u32(w_hi_ptr(s, kc));
          const uint32_t b_lo = b_hi + w_chunk_bytes;
          const int nk = min(kTcBK / 8, p.ksub - kc * (kTcBK / 8));
#pragma unroll
          for (int k = 0; k < kTcBK / 8; ++k) {
            if (k >= nk) break;
            const uint32_t ko = k * 32;
            const uint32_t accum = (kc | k) != 0;
            const uint64_t da = ptx::make_sw128_kmajor_desc(a_hi + ko);
            const uint64_t db = ptx::make_sw128_kmajor_desc(b_hi + ko);
            if (kBf16) {
              ptx::mma_bf16_ss(d_tmem, da, db, idesc, accum);
            } else if (stack_b) {
              ptx::mma_tf32_ss(d_tmem, da, db, idesc2, accum);
              ptx::mma_tf32_ss(c_tmem, ptx::make_sw128_kmajor_desc(a_lo + ko), db, idesc, 1);
            } else if (split) {
              ptx::mma_tf32_ss(c_tmem, ptx::make_sw128_kmajor_desc(a_lo + ko), db, idesc, accum);
              ptx::mma_tf32_ss(c_tmem, da, ptx::make_sw128_kmajor_desc(b_lo + ko), idesc, 1);
              ptx::mma_tf32_ss(d_tmem, da, db, idesc, accum);
            } else {
              ptx::mma_tf32_ss(d_tmem, da, db, idesc, accum);
            }
          }
          YNB_DP_TRACE(3, (int)((tile - blockIdx.x) / gridDim.x), kc);
          ptx::mma_commit(&a_empty[s]);
          if (kc == p.num_chunks - 1) ptx::mma_commit(&tmem_full[acc]);
          if (++s == p.a_stages) { s = 0; ph ^= 1; }
        }
        if (++acc == 2) { acc = 0; acc_ph ^= 1; }
      }
    }
  } else if (warp >= kDpDwWarp0 && warp < kDpDwWarp0 + kDpDwWarps) {
    // ================= depthwise producers: thread = (2x4 output block, 4 channels) =================
    // A chunk is 16 two-row blocks x CGS channel groups = 128 (float) | 256 (bf16) tasks.  bf16: all eight warps work
    // on one chunk.  float: warps 8-11 take the even chunks of this CTA's chunk sequence and warps 12-15 the odd
    // ones — two raw stages are consumed concurrently — so that every thread still owns a two-row block (the rows
    // share two of their three input rows: 24 + 9 shared-memory reads per 8 outputs instead of 2 x (18 + 9); the
    // kernel is bound by the shared-memory pipe, tools/gpu_dp_trace.py + ncu l1tex 70 %).
    constexpr int NGROUPS = kBf16 ? 1 : 2;
    constexpr int GTHREADS = 256 / NGROUPS;
    const int t = (threadIdx.x - kDpDwWarp0 * 32) % GTHREADS;
    const int grp = (threadIdx.x - kDpDwWarp0 * 32) / GTHREADS;
    const int cg = t & (CGS - 1);
    const int IW = TW + 2;
    const bool has_act = p.dw_act != YNB_ACT_NONE;
    const float slope = p.dw_act == YNB_ACT_RELU ? 0.0f : 0.1f;
    const int nloc = (int64_t)blockIdx.x < p.num_tiles
                         ? (int)((p.num_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x) : 0;   // tiles of this CTA
    const int total_chunks = nloc * p.num_chunks;
    bool ok = true;
    {
      for (int gc = grp; gc < total_chunks && ok; gc += NGROUPS) {
        const int lt_ = gc / p.num_chunks, kc = gc - lt_ * p.num_chunks;
        const int r = gc % p.raw_stages, s = gc % p.a_stages;
        const uint32_t rph = (uint32_t)((gc / p.raw_stages) & 1), sph = (uint32_t)((gc / p.a_stages) & 1);
        const float* wv = s_dww + kc * CH + cg * 4;        // this thread's taps: read per filter row (3 x 16 B, broadcast)
        const float4 bv = *reinterpret_cast<const float4*>(wv + 9 * KC);
        ok = ptx::mbar_wait(&raw_full[r], rph, p.err_flag, 7);
        if (ok) ok = ptx::mbar_wait(&a_empty[s], sph ^ 1, p.err_flag, 8);
        if (!ok) break;
        if (t == 0) YNB_DP_TRACE(1, lt_, kc);
        const uint8_t* raw = smem + (size_t)r * lay.raw_stride;
        uint8_t* a_hi = a_stage(s);
        uint8_t* a_lo = a_hi + kTcAStageBytes;
        constexpr int ROWS = 2;
        const int bidx = t / CGS;                          // 0..15
        const int nsx = TW >> 2;
        const int sx = bidx % nsx, sy = (bidx / nsx) * ROWS;
        float4 acc[ROWS][4];
#pragma unroll
        for (int o = 0; o < ROWS; ++o)
#pragma unroll
          for (int q = 0; q < 4; ++q) acc[o][q] = bv;
#pragma unroll
        for (int ir = 0; ir < ROWS + 2; ++ir) {
          const int r0 = (sy + ir) * IW + sx * 4;
          float4 v[6];
#pragma unroll
          for (int j = 0; j < 6; ++j) {
            const int rr = r0 + j;
            if (!kBf16) v[j] = load4(reinterpret_cast<const E*>(raw + rr * 128 + (cg << 4)));
            else v[j] = load4(reinterpret_cast<const E*>(raw + rr * 128 + (cg << 3)));
          }
#pragma unroll
          for (int o = 0; o < ROWS; ++o) {
            const int ky = ir - o;
            if (ky < 0 || ky > 2) continue;
#pragma unroll
            for (int kx = 0; kx < 3; ++kx) {
              const float4 k = *reinterpret_cast<const float4*>(wv + (ky * 3 + kx) * KC);
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                const float4 u = v[q + kx];
                const float2 lo = __ffma2_rn(make_float2(u.x, u.y), make_float2(k.x, k.y), make_float2(acc[o][q].x, acc[o][q].y));
                const float2 hi = __ffma2_rn(make_float2(u.z, u.w), make_float2(k.z, k.w), make_float2(acc[o][q].z, acc[o][q].w));
                acc[o][q] = make_float4(lo.x, lo.y, hi.x, hi.y);
              }
            }
          }
        }
        // the raw tile has been consumed into registers: hand it back before the store phase
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&raw_empty[r]);
#pragma unroll
        for (int o = 0; o < ROWS; ++o) {
          const int row0 = (sy + o) * TW + sx * 4;            // first of this strip's 4 tile rows (= A rows)
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int row = row0 + q;
            float4 a = acc[o][q];
            if (has_act) {
              a.x = fmaxf(a.x, a.x * slope); a.y = fmaxf(a.y, a.y * slope);
              a.z = fmaxf(a.z, a.z * slope); a.w = fmaxf(a.w, a.w * slope);
            }
            if (kBf16) {
              const uint32_t o2 = (uint32_t)row * 128 + ((uint32_t)((cg >> 1) ^ (row & 7)) << 4) + ((uint32_t)(cg & 1) << 3);
              *reinterpret_cast<uint2*>(a_hi + o2) = make_uint2(pack_bf16x2(a.x, a.y), pack_bf16x2(a.z, a.w));
            } else {
              const uint32_t o2 = (uint32_t)row * 128 + ((uint32_t)(cg ^ (row & 7)) << 4);
              if (split) {
                float4 h, l;
                h.x = cvt_rna_tf32(a.x); h.y = cvt_rna_tf32(a.y); h.z = cvt_rna_tf32(a.z); h.w = cvt_rna_tf32(a.w);
                l.x = cvt_rna_tf32(a.x - h.x); l.y = cvt_rna_tf32(a.y - h.y);
                l.z = cvt_rna_tf32(a.z - h.z); l.w = cvt_rna_tf32(a.w - h.w);
                *reinterpret_cast<float4*>(a_hi + o2) = h;
                *reinterpret_cast<float4*>(a_lo + o2) = l;
              } else {
                *reinterpret_cast<float4*>(a_hi + o2) = a;
              }
            }
          }
        }
        ptx::fence_proxy_async_smem();     // generic-proxy writes -> visible to the tensor core
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&a_ready[s]);
        if (t == 0) YNB_DP_TRACE(2, lt_, kc);
      }
    }
  } else if (warp < kDpEpiWarps) {
    // ================= epilogue: two groups of four warps (group g owns accumulator stage g) =================
    // The thread that owns a tile row builds 128 bytes of its OUTPUT row in the warp's swizzled staging box
    // (interleaved with the pass-through half for ShuffleNet units) — no transposition: it owns the same row
    // of the accumulator — and the warp then copies the box out with 16-byte accesses (whole 128-byte row
    // segments per instruction).
    const int group = warp >> 2, q = warp & 3;            // group g drains the tiles with (local index & 1) == g
    const int row = q * 32 + lane;
    const float slope = p.act == YNB_ACT_RELU ? 0.0f : (p.act == YNB_ACT_LEAKY ? 0.1f : 1.0f);
    uint8_t* sbox = smem + lay.stg_off + warp * 4096;
    const int sw = lane & 7;
    const int yy = row >> p.lgTW, xx = row & (TW - 1);
    constexpr int BOX = 128 / (int)sizeof(E);              // output elements per row and box: 32 | 64
    constexpr int CPB = kPass ? BOX / 2 : BOX;             // accumulator columns per box: 16/32 | 32/64
    constexpr int EPC = 16 / (int)sizeof(E);               // elements per 16-byte chunk: 4 | 8
    const int nbox = (p.Npad + CPB - 1) / CPB;
    const int out_cols = kPass ? 2 * p.N : ((p.N + EPC - 1) / EPC) * EPC;   // logical output elements per row
    E* const outp = reinterpret_cast<E*>(p.out);
    const E* const passp = reinterpret_cast<const E*>(p.pass);
    const int acc = group;
    bool ok = true;
    int lt = group;
    for (int64_t tile = blockIdx.x + (int64_t)group * gridDim.x; tile < p.num_tiles && ok; tile += 2 * (int64_t)gridDim.x, lt += 2) {
      const uint32_t acc_ph = (uint32_t)((lt >> 1) & 1);
      const int b = (int)(tile / per_img);
      const int rr = (int)(tile - (int64_t)b * per_img);
      const int y = (rr / p.tiles_x) * TH + yy, x = (rr % p.tiles_x) * TW + xx;
      const bool valid = y < p.H && x < p.W;
      const int pix = (b * p.H + y) * p.W + x;
      const int ooff = valid ? pix * p.out_ld : -1;        // element offsets fit 32 bits (checked at plan time)
      const E* prow = passp + (valid ? (size_t)pix * p.pass_ld : 0);
      uint4 x1v[4];                                        // the CPB pass-through elements of the next box (64 bytes)
      auto fetch_x1 = [&](int c0) {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          x1v[j] = (kPass && valid && c0 + EPC * j < p.N) ? __ldg(reinterpret_cast<const uint4*>(prow + c0) + j)
                                                         : make_uint4(0u, 0u, 0u, 0u);
      };
      if (kPass) fetch_x1(0);
      ok = ptx::mbar_wait(&tmem_full[acc], acc_ph, p.err_flag, 9);
      if (!ok) break;
      ptx::tc_fence_after_sync();
      if (q == 0 && lane == 0) YNB_DP_TRACE(4, lt, 0);
      const uint32_t t_base = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * acc_cols);
      // 16 accumulator columns -> bias -> activation, in registers
      auto drain16 = [&](int c0, float (&v)[16]) {
        uint32_t r1[16];
        ptx::tmem_ld_32x16(t_base + c0, r1);
        if (nacc == 2) {
          uint32_t r2[16];
          ptx::tmem_ld_32x16(t_base + (uint32_t)p.Npad + c0, r2);
          ptx::tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(r1[j]) + __uint_as_float(r2[j]);
        } else {
          ptx::tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(r1[j]);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4 b4 = *reinterpret_cast<const float4*>(s_bias + c0 + 4 * j);
          v[4 * j] += b4.x; v[4 * j + 1] += b4.y; v[4 * j + 2] += b4.z; v[4 * j + 3] += b4.w;
        }
        if (p.act == YNB_ACT_RELU) {
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.0f);
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], v[j] * slope);
        }
      };
      auto put_chunk = [&](int j, uint4 val) {               // 16-byte chunk j of this thread's staging row
        *reinterpret_cast<uint4*>(sbox + lane * 128 + ((j ^ sw) << 4)) = val;
      };
      const bool tma_out = p.tma_out != 0;
      for (int bx = 0; bx < nbox; ++bx) {
        const int c0 = bx * CPB;
        // the previous TMA store of this warp must have finished READING the staging box before it is rewritten:
        // waited for AFTER the first accumulator load of the box, whose latency covers it
        auto box_free = [&]() {
          if (tma_out) {
            if (ptx::elect_one()) ptx::bulk_wait_read<0>();
            __syncwarp();
          }
        };
        if (!kBf16 && kPass) {
          float v[16];
          drain16(c0, v);
          box_free();
          const uint32_t xw[16] = {x1v[0].x, x1v[0].y, x1v[0].z, x1v[0].w, x1v[1].x, x1v[1].y, x1v[1].z, x1v[1].w,
                                   x1v[2].x, x1v[2].y, x1v[2].z, x1v[2].w, x1v[3].x, x1v[3].y, x1v[3].z, x1v[3].w};
#pragma unroll
          for (int j = 0; j < 8; ++j)      // chunk j = (x1[2j], conv[2j], x1[2j+1], conv[2j+1])
            put_chunk(j, make_uint4(xw[2 * j], __float_as_uint(v[2 * j]), xw[2 * j + 1], __float_as_uint(v[2 * j + 1])));
        } else if (!kBf16) {
          float v[16];
          drain16(c0, v);
          box_free();
#pragma unroll
          for (int j = 0; j < 4; ++j)
            put_chunk(j, make_uint4(__float_as_uint(v[4 * j]), __float_as_uint(v[4 * j + 1]), __float_as_uint(v[4 * j + 2]),
                                    __float_as_uint(v[4 * j + 3])));
          if (c0 + 16 < p.Npad) {
            drain16(c0 + 16, v);
#pragma unroll
            for (int j = 0; j < 4; ++j)
              put_chunk(4 + j, make_uint4(__float_as_uint(v[4 * j]), __float_as_uint(v[4 * j + 1]),
                                          __float_as_uint(v[4 * j + 2]), __float_as_uint(v[4 * j + 3])));
          }
        } else if (kPass) {
          box_free();
          // bf16: one 32-bit word per output pair = (x1[i] in the low half, conv[i] in the high half)
          const uint32_t xw[16] = {x1v[0].x, x1v[0].y, x1v[0].z, x1v[0].w, x1v[1].x, x1v[1].y, x1v[1].z, x1v[1].w,
                                   x1v[2].x, x1v[2].y, x1v[2].z, x1v[2].w, x1v[3].x, x1v[3].y, x1v[3].z, x1v[3].w};
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            if (h == 0 || c0 + 16 < p.Npad) {
              float v[16];
              drain16(c0 + 16 * h, v);
              uint32_t w[16];
#pragma unroll
              for (int i = 0; i < 16; ++i) {
                const uint32_t xs = xw[8 * h + (i >> 1)];
                const uint32_t x1bits = (i & 1) ? (xs >> 16) : (xs & 0xffffu);
                w[i] = x1bits | (pack_bf16x2(0.0f, v[i]) & 0xffff0000u);
              }
#pragma unroll
              for (int j = 0; j < 4; ++j) put_chunk(4 * h + j, make_uint4(w[4 * j], w[4 * j + 1], w[4 * j + 2], w[4 * j + 3]));
            }
          }
        } else {
          box_free();
#pragma unroll
          for (int h = 0; h < 4; ++h) {
            if (h == 0 || c0 + 16 * h < p.Npad) {
              float v[16];
              drain16(c0 + 16 * h, v);
              put_chunk(2 * h, make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]),
                                          pack_bf16x2(v[6], v[7])));
              put_chunk(2 * h + 1, make_uint4(pack_bf16x2(v[8], v[9]), pack_bf16x2(v[10], v[11]), pack_bf16x2(v[12], v[13]),
                                              pack_bf16x2(v[14], v[15])));
            }
          }
        }
        if (kPass && bx + 1 < nbox) fetch_x1((bx + 1) * CPB);
        if (bx == nbox - 1) {              // all TMEM reads of this tile are done: hand the stage back
          ptx::tc_fence_before_sync();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&tmem_empty[acc]);
        }
        __syncwarp();
        const int j0 = bx * BOX;           // first logical output element of this box
        if (tma_out) {
          // the warp's 32 tile rows are TW x (32 / TW) pixels of one image: the swizzled box leaves through ONE
          // tensor store, rows outside the image and channels >= the logical width clipped by the copy engine
          ptx::fence_proxy_async_smem();
          __syncwarp();
          if (ptx::elect_one()) {
            ptx::tma_store_4d(&tmOut, sbox, j0, (rr % p.tiles_x) * TW, (rr / p.tiles_x) * TH + q * (32 >> p.lgTW), b);
            ptx::bulk_commit();
          }
          continue;
        }
        // Per-lane copy-out, for outputs the tensor map cannot describe: lanes 0-15 store two 128-byte row segments per
        // instruction.  (Full-warp stores of four rows cost the bf16 instantiations two more registers, CUDA 12.9.)
        const int ch = lane & 7;
        const int jc = j0 + EPC * ch;
#pragma unroll 8
        for (int k = 0; k < 16; ++k) {
          const int r = ((lane >> 3) & 1) + 2 * k;
          const int oo = __shfl_sync(0xffffffffu, ooff, r);
          const uint4 val = *reinterpret_cast<const uint4*>(sbox + r * 128 + ((ch ^ (r & 7)) << 4));
          if (lane < 16 && oo >= 0 && jc < out_cols) *reinterpret_cast<uint4*>(outp + oo + p.out_off + jc) = val;
        }
        __syncwarp();
      }
      if (q == 0 && lane == 0) YNB_DP_TRACE(5, lt, 0);
    }
    if (p.tma_out && ptx::elect_one()) ptx::bulk_wait<0>();     // all output boxes have landed
  }

  ptx::tc_fence_before_sync();
  __syncthreads();
  if (warp == kDpMmaWarp) {
    ptx::tc_fence_after_sync();
    ptx::tmem_dealloc(tmem_base, p.tmem_cols);
  }
}

// --------------------------------------------------------------------------------------
// host side
// --------------------------------------------------------------------------------------
struct DwPwLaunch {
  CUtensorMap tmIn;
  CUtensorMap tmOut;      // valid when p.tma_out
  CUtensorMap tmPass;     // pass-through half (L2 prefetch only); valid when p.pass_blocks > 0
  const TcWeights* w = nullptr;
  DwPwParams p;
  uint32_t smem = 0;
  unsigned grid = 0;
};

// Tile, stages and residency for one fused launch; false = use the unfused pair (shape does not fit).
// in: view [B][H][W][C4 of in_ld] starting at `in` (16-byte aligned), out / pass views likewise.
inline bool plan_dwpw(DwPwLaunch& L, const void* in, int in_ld, int B, int H, int W, int C, int C4, const TcWeights* w,
                      int mode) {
  DwPwParams& p = L.p;
  const bool split = mode == YNB_GEMM_TC_3XTF32;
  const bool is_bf16 = mode == YNB_GEMM_TC_BF16;
  const int es = is_bf16 ? 2 : 4, chunk_ch = 128 / es;
  // TMEM: two accumulator stages of (main [+ corr]) x Npad columns
  if (2 * (split ? 2 : 1) * w->Npad > 512 || (reinterpret_cast<uintptr_t>(in) & 15u) || ((in_ld * es) & 15)) return false;
  if ((int64_t)B * H * W * std::max(p.out_ld, std::max(p.pass_ld, 1)) >= (1LL << 31)) return false;
  p.H = H; p.W = W;
  {   // 16 x 8 or 32 x 4 output pixels per tile: whichever covers the map with fewer tiles
    const int t16 = ((W + 15) / 16) * ((H + 7) / 8), t32 = ((W + 31) / 32) * ((H + 3) / 4);
    p.lgTW = t32 < t16 ? 5 : 4;
  }
  const int TW = 1 << p.lgTW, TH = kTcBM >> p.lgTW;
  p.tiles_x = (W + TW - 1) / TW;
  p.tiles_y = (H + TH - 1) / TH;
  p.num_tiles = (int64_t)B * p.tiles_x * p.tiles_y;
  p.C4 = C4;
  p.num_chunks = w->Kpad / chunk_ch;
  p.ksub = (C * es + 31) / 32;            // valid 32-byte K sub-steps (8 tf32 | 16 bf16 per MMA)
  p.N = w->N; p.Npad = w->Npad;
  p.mode = mode;
  p.tmem_cols = 32;
  while ((int)p.tmem_cols < 2 * (split ? 2 : 1) * p.Npad) p.tmem_cols <<= 1;
  // Shared memory: a 2-deep A ring is enough (it only decouples the depthwise producers from the MMAs, both
  // on chip); everything else goes to the raw ring — the TMA bytes in flight per SM are what bounds the HBM rate.
  bool found = false;
  for (int raw = kDpMaxRawStages; raw >= 2 && !found; --raw)
    for (int resident = 1; resident >= 0 && !found; --resident) {
      DpSmemLayout lay = dp_smem_layout(p.Npad, p.num_chunks, p.lgTW, 2, raw, resident != 0, split, chunk_ch);
      if (lay.total <= (uint32_t)kTcSmemBudget) {
        p.a_stages = 2; p.raw_stages = raw; p.w_resident = resident; L.smem = lay.total;
        found = true;
      }
    }
  if (!found) return false;
  const int epc = 16 / es;                // elements per 16 bytes
  if ((reinterpret_cast<uintptr_t>(p.out) & 15u) || (p.out_ld % epc) || (p.out_off % epc)) return false;
  p.pass_blocks = 0;
  if (p.pass) {
    if ((reinterpret_cast<uintptr_t>(p.pass) & 15u) || (p.pass_ld % epc)) return false;
    if (make_tmap_nhwc(&L.tmPass, p.pass, (p.N + epc - 1) / epc * epc, W, H, B, p.pass_ld, TW, TH, is_bf16))
      p.pass_blocks = (p.N + chunk_ch - 1) / chunk_ch;
  }
  // the raw tile is NOT swizzled: the depthwise threads that read one tile row together cover its 128 bytes
  // (lane = channel group fastest), so plain rows are conflict-free and need no XOR per load
  if (!make_tmap_nhwc(&L.tmIn, in, C4, W, H, B, in_ld, TW + 2, TH + 2, is_bf16, false)) return false;
  {
    const int out_cols = p.pass ? 2 * p.N : (p.N + epc - 1) / epc * epc;
    p.tma_out = p.out_off == 0 && make_tmap_nhwc(&L.tmOut, p.out, out_cols, W, H, B, p.out_ld, TW, 32 / TW, is_bf16);
  }
  L.w = w;
  L.grid = (unsigned)std::min<int64_t>(p.num_tiles, kNumSMs);
  return true;
}

inline cudaError_t launch_dwpw_tc(const DwPwLaunch& L, cudaStream_t st) {
  using KernelT = void (*)(CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, DwPwParams);
  static const KernelT kernels[4] = {dwpw_tc_kernel<false, float>, dwpw_tc_kernel<true, float>,
                                     dwpw_tc_kernel<false, bf16>, dwpw_tc_kernel<true, bf16>};
  static bool attr_set = false;
  if (!attr_set) {
    for (KernelT k : kernels) {
      cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, kTcSmemBudget);
      if (e != cudaSuccess) return e;
    }
    attr_set = true;
  }
  const int ki = (L.p.mode == YNB_GEMM_TC_BF16 ? 2 : 0) + (L.p.pass != nullptr ? 1 : 0);
  cudaError_t r = launch_pdl(kernels[ki], dim3(L.grid), dim3(kDpThreads), (size_t)L.smem, st,
                             L.tmIn, L.w->tm_hi, L.w->tm_lo, L.p.pass_blocks ? L.tmPass : L.tmIn,
                             L.p.tma_out ? L.tmOut : L.tmIn, L.p);
  YNB_COUNT_LAUNCH();
  return r;
}

}  // namespace ynb
