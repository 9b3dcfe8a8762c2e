// C ABI of the B200-native YOLO-Nano forward path (include/yolonano_b200.h):
// engine lifecycle, weight packing, workspace planning and the per-batch launch plan.
#include <cuda.h>
#include <cuda_runtime.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <functional>
#include <map>
#include <memory>
#include <string>
#include <tuple>
#include <vector>

#include "yolonano_b200.h"

#include "common.cuh"
#include "decode_nms.cuh"
#include "nms_grid.cuh"
#include "gemm_ffma.cuh"
#include "gemm_tc.cuh"
#include "unit_tc.cuh"
#include "kernels_basic.cuh"
#include "train_ops.cuh"
#include "wgrad_tc.cuh"
#include "voc_eval.cuh"
#include "coco_eval.cuh"
#include "topology.h"

#define YNB_EXPORT extern "C" __attribute__((visibility("default")))

namespace ynb {

thread_local LaunchCounter* g_counter = nullptr;
static thread_local std::string g_create_error;

// Physical NHWC tensor in the workspace.
struct Tensor {
  float* p = nullptr;   // base address (element type: float, or bf16 when es == 2 — use at())
  int es = 4;       // element size in bytes
  int C = 0;        // logical channels
  int ld = 0;       // elements per pixel
  int H = 0, W = 0;
  size_t floats_per_image() const { return (size_t)H * W * ld; }
  void* at(int off = 0) const { return reinterpret_cast<char*>(p) + (size_t)off * es; }   // address of element `off`
};

// How a conv's input channels are laid out physically (static per conv).
struct InLayout {
  int ktot;       // physical width read by the conv (multiple of 4)
  int shift;      // logical input channel k sits at position k + shift of the view
};

struct PackedConv {
  bool loaded = false;
  std::vector<float> w_host, b_host;   // reference layout [cout][cin/g][k][k], [cout]
  float* w_dev = nullptr;              // FFMA / dw / stem layout
  float* b_dev = nullptr;
  int n = 0, ktot = 0;                 // GEMM dims of the packed matrix
  TcWeights tc;                        // tensor-core layout (dense convs only)
};

// One kernel launch of the plan, with what bench.py needs for the roofline: a label, the
// kernel family, and its ALGORITHMIC bytes / flops (unique unpadded inputs + outputs +
// weights; DESIGN.md "algorithmic bytes").
struct Op {
  std::string name, kind;
  double bytes = 0, flops = 0;
  std::function<cudaError_t(cudaStream_t)> fn;
  bool mark = false;   // record a fork point on the main stream BEFORE this op
  bool side = false;   // runs on the side stream, after the most recent fork point
  bool join = false;   // main stream waits for the last side op before this op
};

struct ProfEntry {
  std::string name, kind;
  double bytes, flops;
  float ms;
};

struct Plan {
  int batch = 0;
  std::vector<Op> net;        // stem .. the last hidden conv of every head
  std::vector<Op> raw_tail;   // head_det_*.4 -> raw maps (ynb_forward_raw, FFMA mode, odd class counts)
  std::vector<Op> decode;     // raw -> boxes/scores/cls (engine buffers), after raw_tail
  std::vector<Op> fused_tail; // head_det_*.4 with the decode in the GEMM epilogue: no raw map
  bool fused = false;
};

}  // namespace ynb

using namespace ynb;

struct ynb_engine {
  ynb_config cfg;
  int S = 0;
  std::string err;
  std::vector<ConvSpec> table;
  std::map<std::string, int> index;
  std::vector<PackedConv> convs;
  // merged (branch1.2 | branch2.5) pointwise convs of the three stride-2 units, split along N when wider than one
  // MMA tile: cat[stage][part]; K = [branch1 dw output | branch2 dw output], rows = interleaved output slots
  struct CatConv { PackedConv pc; int n0 = 0, k1p = 0, k2p = 0; };
  std::vector<CatConv> cat[3];
  StemWeights stem_w;                      // folded stem weights, passed as a kernel parameter
  PreLut prelut;                           // uint8 -> normalised float32 table (ynb_set_normalization)
  PreLut* d_prelut = nullptr;              // its device copy
  struct StemMap { CUtensorMap tm; int ok; };
  std::map<std::tuple<const float*, int, int>, StemMap> stem_maps;   // TMA maps over caller inputs, by (pointer, batch, S)
  bool committed = false;

  // workspace
  char* ws = nullptr;
  size_t ws_bytes = 0;
  int ws_batch = 0, ws_S = 0;
  std::map<std::string, Tensor> taps;      // name -> tensor (also used by the planner)
  Tensor raw[3];
  float* d_boxes = nullptr;
  float* d_scores = nullptr;
  int32_t* d_cls = nullptr;
  void* d_nms_ws = nullptr;
  int64_t nms_ws_bytes = 0;
  // host-call staging
  float* d_x = nullptr;                // == slot[0].x
  struct HostSlot {                    // double-buffered host I/O (ynb_submit_host / ynb_wait_host)
    float* x = nullptr; float* boxes = nullptr; float* scores = nullptr; int32_t* cls = nullptr;
    int32_t* counts = nullptr;
    uint8_t* img_u8 = nullptr;         // [B,S,S,3] staging for the uint8 entry
    int32_t* rects = nullptr;          // [B][4]
    cudaEvent_t h2d = nullptr, done = nullptr;
    bool busy = false;
    int batch = 0;
    float* ob = nullptr; float* os = nullptr; int32_t* oc = nullptr; int32_t* on = nullptr;   // host destinations
    int* flag_host = nullptr;          // pinned: device error word of this step
  } slot[2];
  cudaStream_t s_copy = nullptr;       // H2D next to the compute stream
  cudaStream_t s_copy2 = nullptr;      // second half of a large H2D (two DMA queues: 53 -> 55 GB/s measured)
  cudaEvent_t ev_copy2 = nullptr;
  cudaStream_t s_d2h = nullptr;        // results back to the host (PCIe is full duplex: its own stream)
  const float* d_x_bound = nullptr;   // input of the forward in flight
  float* d_out_boxes = nullptr;
  float* d_out_scores = nullptr;
  int32_t* d_out_cls = nullptr;
  int32_t* d_out_counts = nullptr;
  int* d_err = nullptr;

  std::map<int, std::unique_ptr<Plan>> plans;
  std::deque<std::deque<TcGemmLaunch>> tc_store;
  std::deque<std::deque<DwPwLaunch>> dp_store;   // fused depthwise -> pointwise launches
  std::deque<CUtensorMap> dw_maps;         // input maps of the depthwise launches (stable addresses)

  // execution resources: all engine work runs on the engine's own streams, ordered against
  // the caller's stream with events (stream capture is not allowed on the legacy stream)
  cudaStream_t s_main = nullptr, s_side = nullptr;
  std::vector<cudaEvent_t> events;
  size_t ev_next = 0;
  cudaEvent_t ev_in = nullptr, ev_out = nullptr;
  struct GraphKey {
    int batch; const void* x; const void* ob; const void* os; const void* oc; const void* on;
    float conf, thr; int diou, mode, S;
    bool operator<(const GraphKey& o) const {
      return std::tie(batch, x, ob, os, oc, on, conf, thr, diou, mode, S) <
             std::tie(o.batch, o.x, o.ob, o.os, o.oc, o.on, o.conf, o.thr, o.diou, o.mode, o.S);
    }
  };
  std::map<GraphKey, cudaGraphExec_t> graphs;
  std::map<GraphKey, int> graph_seen;
  bool use_graphs = true;
  std::map<int, int64_t> graph_launches;   // kernel launches inside one captured forward, per batch
  LaunchCounter counter;
  bool profiling = false;
  std::vector<ProfEntry> prof;

  int64_t N() const {
    int64_t n = 0;
    for (int s : {8, 16, 32}) n += (int64_t)cfg.num_anchors * (S / s) * (S / s);
    return n;
  }
};

namespace ynb {
inline bool is_bf16(const ynb_engine* e) { return e->cfg.gemm_mode == YNB_GEMM_TC_BF16; }
}  // namespace ynb

namespace {

int fail(ynb_engine* e, int code, const std::string& msg) {
  if (e) e->err = msg; else g_create_error = msg;
  return code;
}
#define CUDA_TRY(e, call)                                                                 \
  do {                                                                                    \
    cudaError_t _st = (call);                                                             \
    if (_st != cudaSuccess)                                                               \
      return fail(e, YNB_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(_st));  \
  } while (0)

struct CounterScope {
  explicit CounterScope(ynb_engine* e) { g_counter = &e->counter; }
  ~CounterScope() { g_counter = nullptr; }
};

// ---- static layout knowledge -----------------------------------------------------------
// TMA views and 16-byte loads must start 16-byte aligned: 4 floats or 8 bf16.  Stage outputs are DENSE (float stage 2:
// 116 channels; bf16 stage 2: 116 + 4 zero pad, stage 3: 232), any pad at the END of the row.  Where the second half
// does not start on a 16-byte boundary (h = 58 floats, 58 / 116 bf16), the one conv that reads only x2 (branch2[0] of
// the stride-1 units) reads the aligned window that starts h % a channels earlier, with its weights shifted by as many
// input positions (zero weight on the leading channels): see x2_window() / in_layout().  A dense layout lets the fused
// unit tails leave through TMA tensor stores.
int stage_ld(bool bf, int si) { return round_up(stage_channels()[si + 1], bf ? 8 : 4); }
// Aligned window over the second half of a stage output: start channel and weight shift.
struct X2Window { int off, shift; };
X2Window x2_window(int h, int a) { return {h - h % a, h % a}; }

// Input layout of conv `name` (see plan_network for the producers).
InLayout in_layout(const ConvSpec& c, bool bf) {
  const std::string& n = c.name;
  if (c.kind == kDense3x3) return {c.cin == 3 ? 27 : 9 * c.cin, 0};
  bool reads_c3 = n == "backbone.stage3.0.branch1.0" || n == "backbone.stage3.0.branch1.2" ||
                  n == "backbone.stage3.0.branch2.0" || n == "conv1x1_0.convs.0";
  bool reads_c4 = n == "backbone.stage4.0.branch1.0" || n == "backbone.stage4.0.branch1.2" ||
                  n == "backbone.stage4.0.branch2.0" || n == "conv1x1_1.convs.0";
  if (reads_c3) return {stage_ld(bf, 0), 0};
  if (reads_c4) return {stage_ld(bf, 1), 0};
  // branch2[0] of a stride-1 unit reads x2 of its stage's output: through an aligned, shifted window
  for (int si = 0; si < 3; ++si) {
    const std::string pre = "backbone.stage" + std::to_string(si + 2) + ".";
    if (n.compare(0, pre.size(), pre) == 0 && n.size() > pre.size() + 2 && n[pre.size()] != '0' &&
        n.compare(n.size() - 10, 10, ".branch2.0") == 0) {
      const int a = bf ? 8 : 4;
      const X2Window w = x2_window(c.cin, a);
      if (w.shift) return {round_up(c.cin + w.shift, a), w.shift};
    }
  }
  return {round_up(c.cin, bf ? 8 : 4), 0};
}

// ---- weight packing ----------------------------------------------------------------------
// Packs a dense [n][ktot] fp32 matrix (ktot = taps x kin) for the tensor-core path of the engine's mode:
//   fp32 modes: [Npad][Kpad] split into exact-tf32 hi and lo planes, K chunks of 32;
//   bf16 mode : ONE plane of bf16 (round to nearest even), K chunks of 64; a 3x3 conv pads every tap to whole chunks
//               ([N][tap][128] for 96 channels) so that a K step never straddles two taps.
int pack_tc_matrix(ynb_engine* e, TcWeights& t, const float* w, int n, int ktot, int taps, const std::string& name) {
  const bool bf = is_bf16(e);
  t.N = n;
  t.Npad = round_up(n, 16);
  if (t.hi) cudaFree(t.hi);
  if (t.lo) cudaFree(t.lo);
  if (t.bw) cudaFree(t.bw);
  t.hi = t.lo = nullptr; t.bw = nullptr;
  if (bf) {
    const int kin = ktot / taps, kin_pad = round_up(kin, 64);
    t.Kpad = taps * kin_pad;
    std::vector<bf16> bw((size_t)t.Npad * t.Kpad, __float2bfloat16(0.0f));
    for (int r = 0; r < n; ++r)
      for (int tp = 0; tp < taps; ++tp)
        for (int k = 0; k < kin; ++k)
          bw[(size_t)r * t.Kpad + (size_t)tp * kin_pad + k] = __float2bfloat16_rn(w[(size_t)r * ktot + (size_t)tp * kin + k]);
    CUDA_TRY(e, cudaMalloc(&t.bw, bw.size() * 2));
    CUDA_TRY(e, cudaMemcpy(t.bw, bw.data(), bw.size() * 2, cudaMemcpyHostToDevice));
    if (!make_tmap_2d(&t.tm_hi, t.bw, t.Kpad, t.Npad, t.Kpad, t.Npad, true))
      return fail(e, YNB_ERR_CUDA, "cuTensorMapEncodeTiled failed for weights of " + name);
    t.tm_lo = t.tm_hi;
    return YNB_OK;
  }
  t.Kpad = round_up(ktot, kTcBK);
  std::vector<float> hi((size_t)t.Npad * t.Kpad, 0.f), lo((size_t)t.Npad * t.Kpad, 0.f);
  for (int r = 0; r < n; ++r)
    for (int k = 0; k < ktot; ++k)
      split_tf32_host(w[(size_t)r * ktot + k], &hi[(size_t)r * t.Kpad + k], &lo[(size_t)r * t.Kpad + k]);
  CUDA_TRY(e, cudaMalloc(&t.hi, hi.size() * 4));
  CUDA_TRY(e, cudaMalloc(&t.lo, lo.size() * 4));
  CUDA_TRY(e, cudaMemcpy(t.hi, hi.data(), hi.size() * 4, cudaMemcpyHostToDevice));
  CUDA_TRY(e, cudaMemcpy(t.lo, lo.data(), lo.size() * 4, cudaMemcpyHostToDevice));
  if (!make_tmap_2d(&t.tm_hi, t.hi, t.Kpad, t.Npad, t.Kpad, t.Npad) ||
      !make_tmap_2d(&t.tm_lo, t.lo, t.Kpad, t.Npad, t.Kpad, t.Npad))
    return fail(e, YNB_ERR_CUDA, "cuTensorMapEncodeTiled failed for weights of " + name);
  return YNB_OK;
}

// The two output branches of a stride-2 ShuffleNetV2 unit as ONE pointwise conv (backbone/shufflenetv2.py:43-49,
// 57-63, 73-76): A = [branch1 dw output | branch2 dw output] concatenated along K (each padded to whole K chunks),
// weights block-diagonal with the rows interleaved the way channel_shuffle interleaves the branches:
//   row 2i = [ W_branch1.2[i] | 0 ],   row 2i+1 = [ 0 | W_branch2.5[i] ]      (+ zero rows on the pad at the end)
// so that torch.cat + channel_shuffle is the GEMM's plain dense output (TMA-store epilogue) instead of two launches
// with 4-byte scattered stores.  Wider than one MMA tile (stage 4: 464 columns) -> split along N.
int pack_cat(ynb_engine* e, int si) {
  const bool bf = is_bf16(e);
  const std::string bk = "backbone.stage" + std::to_string(si + 2) + ".0.";
  const int i1 = e->index.at(bk + "branch1.2"), i2 = e->index.at(bk + "branch2.5");
  const ConvSpec& c1 = e->table[i1];
  const ConvSpec& c2 = e->table[i2];
  const PackedConv& p1 = e->convs[i1];
  const PackedConv& p2 = e->convs[i2];
  const InLayout il1 = in_layout(c1, bf), il2 = in_layout(c2, bf);
  const int ld = stage_ld(bf, si);
  const int ch = bf ? 64 : kTcBK;
  const int k1p = round_up(il1.ktot, ch), k2p = round_up(il2.ktot, ch), ktot = k1p + k2p;
  const int h = c1.cout;
  std::vector<float> w((size_t)ld * ktot, 0.f), b((size_t)ld, 0.f);
  for (int i = 0; i < h; ++i) {
    const int r1 = 2 * i, r2 = 2 * i + 1;
    for (int k = 0; k < c1.cin; ++k) w[(size_t)r1 * ktot + k + il1.shift] = p1.w_host[(size_t)i * c1.cin + k];
    for (int k = 0; k < c2.cin; ++k) w[(size_t)r2 * ktot + k1p + k + il2.shift] = p2.w_host[(size_t)i * c2.cin + k];
    b[r1] = p1.b_host[i];
    b[r2] = p2.b_host[i];
  }
  const int parts = (ld + 239) / 240;                       // N <= 240 per launch (TMEM: 2 x 240 columns in parity mode)
  const int npart = round_up((ld + parts - 1) / parts, bf ? 8 : 4);
  for (auto& cc : e->cat[si]) {
    if (cc.pc.b_dev) cudaFree(cc.pc.b_dev);
    if (cc.pc.tc.hi) cudaFree(cc.pc.tc.hi);
    if (cc.pc.tc.lo) cudaFree(cc.pc.tc.lo);
    if (cc.pc.tc.bw) cudaFree(cc.pc.tc.bw);
  }
  e->cat[si].clear();
  e->cat[si].resize(parts);
  for (int pi = 0; pi < parts; ++pi) {
    ynb_engine::CatConv& cc = e->cat[si][pi];
    cc.n0 = pi * npart;
    const int n = std::min(npart, ld - cc.n0);
    cc.k1p = k1p; cc.k2p = k2p;
    cc.pc.n = n; cc.pc.ktot = ktot; cc.pc.loaded = true;
    CUDA_TRY(e, cudaMalloc(&cc.pc.b_dev, round_up(n, 4) * 4));
    CUDA_TRY(e, cudaMemset(cc.pc.b_dev, 0, round_up(n, 4) * 4));
    CUDA_TRY(e, cudaMemcpy(cc.pc.b_dev, b.data() + cc.n0, n * 4, cudaMemcpyHostToDevice));
    // the K blocks are already padded to whole chunks: pack as ONE tap of width ktot
    int rc = pack_tc_matrix(e, cc.pc.tc, w.data() + (size_t)cc.n0 * ktot, n, ktot, 1, bk + "cat");
    if (rc) return rc;
  }
  return YNB_OK;
}

int pack_conv(ynb_engine* e, int i) {
  const ConvSpec& c = e->table[i];
  PackedConv& pc = e->convs[i];
  const bool bf = is_bf16(e);
  InLayout il = in_layout(c, bf);
  std::vector<float> w, b;
  if (c.kind == kDense3x3 && c.cin == 3) {            // stem: [27][24]
    w.assign(27 * 24, 0.f);
    for (int co = 0; co < 24; ++co)
      for (int ci = 0; ci < 3; ++ci)
        for (int t = 0; t < 9; ++t) w[(ci * 9 + t) * 24 + co] = pc.w_host[(co * 3 + ci) * 9 + t];
    b = pc.b_host;
    pc.n = 24; pc.ktot = 27;
    memcpy(e->stem_w.w, w.data(), sizeof(e->stem_w.w));
    memcpy(e->stem_w.b, b.data(), sizeof(e->stem_w.b));
  } else if (c.kind == kDw3x3) {                       // [9][C4] by physical position
    int c4 = il.ktot;
    w.assign(9 * c4, 0.f);
    b.assign(c4, 0.f);
    for (int ch = 0; ch < c.cin; ++ch) {
      int s = ch + il.shift;
      for (int t = 0; t < 9; ++t) w[t * c4 + s] = pc.w_host[ch * 9 + t];
      b[s] = pc.b_host[ch];
    }
    pc.n = c4; pc.ktot = 9;
  } else if (c.kind == kPw1x1) {                       // [N][Ktot] by physical position
    w.assign((size_t)c.cout * il.ktot, 0.f);
    for (int n = 0; n < c.cout; ++n)
      for (int k = 0; k < c.cin; ++k) w[(size_t)n * il.ktot + k + il.shift] = pc.w_host[(size_t)n * c.cin + k];
    b = pc.b_host;
    pc.n = c.cout; pc.ktot = il.ktot;
  } else {                                             // dense 3x3: [N][tap][cin]
    w.assign((size_t)c.cout * 9 * c.cin, 0.f);
    for (int n = 0; n < c.cout; ++n)
      for (int ci = 0; ci < c.cin; ++ci)
        for (int t = 0; t < 9; ++t)
          w[((size_t)n * 9 + t) * c.cin + ci] = pc.w_host[((size_t)n * c.cin + ci) * 9 + t];
    b = pc.b_host;
    pc.n = c.cout; pc.ktot = 9 * c.cin;
  }
  if (pc.w_dev) cudaFree(pc.w_dev);
  if (pc.b_dev) cudaFree(pc.b_dev);
  pc.w_dev = pc.b_dev = nullptr;
  CUDA_TRY(e, cudaMalloc(&pc.w_dev, w.size() * 4));
  CUDA_TRY(e, cudaMalloc(&pc.b_dev, round_up((int)b.size(), 4) * 4));
  CUDA_TRY(e, cudaMemcpy(pc.w_dev, w.data(), w.size() * 4, cudaMemcpyHostToDevice));
  CUDA_TRY(e, cudaMemset(pc.b_dev, 0, round_up((int)b.size(), 4) * 4));
  CUDA_TRY(e, cudaMemcpy(pc.b_dev, b.data(), b.size() * 4, cudaMemcpyHostToDevice));

  // tensor-core layout for the dense contractions (not the stem: K = 27 is HBM-bound)
  if ((c.kind == kPw1x1) || (c.kind == kDense3x3 && c.cin != 3)) {
    int rc = pack_tc_matrix(e, pc.tc, w.data(), pc.n, pc.ktot, c.kind == kDense3x3 ? 9 : 1, c.name);
    if (rc) return rc;
  }
  return YNB_OK;
}

// ---- workspace ---------------------------------------------------------------------------
struct Bump {
  size_t off = 0;
  size_t take(size_t bytes) {
    size_t o = off;
    off += (bytes + 1023) & ~(size_t)1023;
    return o;
  }
};

// Declares every tensor of the forward pass for (batch, S); with base == nullptr it only
// measures.  Keep in sync with plan_network.
size_t layout_workspace(ynb_engine* e, int batch, int S, char* base) {
  Bump bump;
  const bool bf = is_bf16(e);
  const int es_act = bf ? 2 : 4, al = bf ? 8 : 4;
  auto tensor = [&](const std::string& name, int C, int ld, int H, int es = 0) {
    Tensor t;
    t.es = es ? es : es_act;
    t.C = C; t.ld = ld; t.H = H; t.W = H;
    size_t o = bump.take((size_t)batch * H * H * ld * t.es);
    t.p = base ? reinterpret_cast<float*>(base + o) : nullptr;
    e->taps[name] = t;
    return t;
  };
  e->taps.clear();
  const int H1 = S / 4;
  tensor("pool", 24, 24, H1);
  int hin = H1;
  int ld_in = 24;
  for (int si = 0; si < 3; ++si) {
    int cout = stage_channels()[si + 1], h = cout / 2, cin = stage_channels()[si];
    int hout = hin / 2;
    std::string st = "stage" + std::to_string(si + 2);
    const int ld = stage_ld(bf, si);
    int ld_h = round_up(h, al);
    tensor(st + ".b1dw", cin, ld_in, hout);                                    // branch1 dw output (layout of its input)
    tensor(st + ".b2pw", h, ld_h, hin);                                        // branch2 first pw @ input res
    tensor(st + ".mid1", h, ld_h, hout);                                       // pw1 / dw scratch
    tensor(st + ".mid2", h, ld_h, hout);
    for (int bi = 0; bi < stage_repeats()[si]; ++bi) tensor(st + "." + std::to_string(bi), cout, ld, hout);
    hin = hout;
    ld_in = ld;
  }
  const int H3 = S / 8, H4 = S / 16, H5 = S / 32;
  const int hs[3] = {H3, H4, H5};
  for (int l = 0; l < 3; ++l) tensor("lat" + std::to_string(l + 3), 96, 96, hs[l]);
  tensor("sum4", 96, 96, H4); tensor("sum4.lo", 96, 96, H4); tensor("fpn4", 96, 96, H4);
  tensor("sum3", 96, 96, H3); tensor("sum3.lo", 96, 96, H3); tensor("p3", 96, 96, H3);
  tensor("sum4b", 96, 96, H4); tensor("sum4b.lo", 96, 96, H4); tensor("p4", 96, 96, H4);
  tensor("sum5", 96, 96, H5); tensor("sum5.lo", 96, 96, H5); tensor("p5", 96, 96, H5);
  const int ch = e->cfg.num_anchors * (1 + e->cfg.num_classes + 4);
  const char* pn[3] = {"pred_s", "pred_m", "pred_l"};
  for (int l = 0; l < 3; ++l) {
    tensor("head" + std::to_string(l) + ".a", 96, 96, hs[l]);
    tensor("head" + std::to_string(l) + ".b", 96, 96, hs[l]);
    tensor("head" + std::to_string(l) + ".c", 96, 96, hs[l]);
    e->raw[l] = tensor(pn[l], ch, round_up(ch, 4), hs[l], 4);    // raw head maps stay float32
  }
  // aliases used as taps
  e->taps["c3"] = e->taps["stage2.3"];
  e->taps["c4"] = e->taps["stage3.7"];
  e->taps["c5"] = e->taps["stage4.3"];

  int64_t n = 0;
  for (int s : {8, 16, 32}) n += (int64_t)e->cfg.num_anchors * (S / s) * (S / s);
  auto raw = [&](size_t bytes) { size_t o = bump.take(bytes); return base ? base + o : nullptr; };
  e->d_boxes = (float*)raw((size_t)batch * n * 16);
  e->d_scores = (float*)raw((size_t)batch * n * 4);
  e->d_cls = (int32_t*)raw((size_t)batch * n * 4);
  e->nms_ws_bytes = std::max(nms_workspace_bytes(batch, n), grid_nms_workspace_bytes(batch, n));
  e->d_nms_ws = raw((size_t)e->nms_ws_bytes);
  for (int k = 0; k < 2; ++k) {
    e->slot[k].x = (float*)raw((size_t)batch * 3 * S * S * 4);
    e->slot[k].boxes = (float*)raw((size_t)batch * n * 16);
    e->slot[k].scores = (float*)raw((size_t)batch * n * 4);
    e->slot[k].cls = (int32_t*)raw((size_t)batch * n * 4);
    e->slot[k].counts = (int32_t*)raw((size_t)batch * 4);
    e->slot[k].img_u8 = (uint8_t*)raw((size_t)batch * 3 * S * S);
    e->slot[k].rects = (int32_t*)raw((size_t)batch * 16);
  }
  e->d_x = e->slot[0].x;
  e->d_out_boxes = e->slot[0].boxes;
  e->d_out_scores = e->slot[0].scores;
  e->d_out_cls = e->slot[0].cls;
  e->d_out_counts = e->slot[0].counts;
  e->d_err = (int*)raw(256);
  return bump.off;
}

int ensure_workspace(ynb_engine* e, int batch) {
  if (e->ws && e->ws_batch >= batch && e->ws_S == e->S) return YNB_OK;
  int nb = std::max(batch, std::max(e->ws_batch, (int)e->cfg.max_batch));
  CUDA_TRY(e, cudaDeviceSynchronize());
  e->plans.clear();
  e->tc_store.clear(); e->dp_store.clear(); e->dw_maps.clear(); e->stem_maps.clear();
  for (auto& kv : e->graphs) cudaGraphExecDestroy(kv.second);
  e->graphs.clear();
  e->graph_seen.clear();
  if (e->ws) { cudaFree(e->ws); e->ws = nullptr; }
  size_t bytes = layout_workspace(e, nb, e->S, nullptr);
  CUDA_TRY(e, cudaMalloc(&e->ws, bytes));
  // zero once: channel pads (58->60, the pad at the end of a bf16 stage-2 row) are never written afterwards and must be 0
  CUDA_TRY(e, cudaMemset(e->ws, 0, bytes));
  layout_workspace(e, nb, e->S, e->ws);
  e->ws_bytes = bytes;
  e->ws_batch = nb;
  e->ws_S = e->S;
  return YNB_OK;
}

// ---- plan ----------------------------------------------------------------------------------
struct Planner {
  ynb_engine* e;
  int B;
  Plan* plan;
  std::deque<TcGemmLaunch>* tc;
  std::deque<DwPwLaunch>* dp;
  std::string error;
  std::vector<Op>* dst = nullptr;   // op list under construction (defaults to plan->net)
  std::vector<Op>& ops() { return dst ? *dst : plan->net; }

  const PackedConv& conv(const std::string& name) const { return e->convs[e->index.at(name)]; }
  const ConvSpec& spec(const std::string& name) const { return e->table[e->index.at(name)]; }
  Tensor T(const std::string& name) const { return e->taps.at(name); }

  void dw(const std::string& name, const Tensor& in, int in_off, const Tensor& out) {
    const PackedConv& pc = conv(name);
    const ConvSpec& c = spec(name);
    int B_ = B, c4 = pc.n, stride = c.stride, act = c.act;
    const float *w = pc.w_dev, *b = pc.b_dev;
    double px_in = (double)B * in.H * in.W, px_out = (double)B * out.H * out.W;
    const bool bf = is_bf16(e);
    const double bytes = (double)in.es * c.cin * (px_in + px_out) + 40.0 * c.cin, flops = 18.0 * c.cin * px_out;
    // product path: halo tiles through TMA; register-tiled global loads if the view is not 16-byte aligned
    e->dw_maps.emplace_back();
    CUtensorMap* tm = &e->dw_maps.back();
    if (make_tmap_dw(tm, in.p, in.ld, in_off, B, in.H, in.W, c4, stride, bf)) {
      plan->net.push_back({name, "dwconv3x3", bytes, flops, [=](cudaStream_t st) {
        return launch_dwconv3x3_tma(*tm, out.p, out.ld, 0, w, b, B_, in.H, in.W, c4, stride, act, st, false, bf);
      }});
      return;
    }
    if (bf) { error = "bf16 depthwise conv needs a 16-byte aligned view: " + name; return; }
    plan->net.push_back({name, "dwconv3x3", bytes, flops, [=](cudaStream_t st) {
      return launch_dwconv3x3(in.p, in.ld, in_off, out.p, out.ld, 0, w, b, B_, in.H, in.W, c4, stride, act, st);
    }});
  }

  // Pass-through half of a stride-1 unit: out[2i] = x[i].  HBM-bound copy that only
  // depends on the previous unit, so it runs on the side stream next to the unit's convs.
  void passthrough(const std::string& name, const Tensor& x, const Tensor& out, int half) {
    int64_t M = (int64_t)B * x.H * x.W;
    Tensor ps = x, o = out;
    Op op{name + "+passthrough", "interleave_copy", 8.0 * M * half, 0.0, [=](cudaStream_t st) {
      return launch_interleave_copy(ps.p, ps.ld, o.p, o.ld, M, half, st);
    }};
    op.side = true;
    plan->net.push_back(op);
  }

  // pointwise conv: in view (off, ktot) -> out (off, step)
  // `pass`: stride-1 unit tail — out[2i] = pass[i], out[2i+1] = conv[i]
  void pw(const std::string& name, const Tensor& in, int in_off, const Tensor& out, int out_off, int out_step,
          bool join = false, const Tensor* pass = nullptr, const TcGemmParams::Decode* dec = nullptr) {
    const PackedConv& pc = conv(name);
    const ConvSpec& c = spec(name);
    int64_t M = (int64_t)B * in.H * in.W;
    const bool tc_mode = e->cfg.gemm_mode != YNB_GEMM_FP32_FFMA;
    const bool bf = is_bf16(e);
    const double abytes = (double)in.es * M * c.cin + (double)out.es * M * (c.cout + (pass && tc_mode ? 2.0 * c.cout : 0.0)) +
                          (bf ? 2.0 : 4.0) * c.cin * c.cout + 4.0 * c.cout;
    const double aflops = 2.0 * M * c.cin * c.cout;
    if (e->cfg.gemm_mode == YNB_GEMM_FP32_FFMA) {
      GemmParams g{};
      g.a = in.p; g.a_ld = in.ld; g.a_off = in_off; g.a2 = nullptr; g.a2_mode = 0;
      g.w = pc.w_dev; g.bias = pc.b_dev; g.out = out.p; g.out_ld = out.ld;
      g.out_off = out_off; g.out_step = out_step;
      g.M = M; g.N = pc.n; g.Ktot = pc.ktot; g.act = c.act;
      if (pass) { g.out_off = 1; g.out_step = 2; }
      Op op{name, "pw_ffma", abytes, aflops, [=](cudaStream_t st) { return launch_gemm_ffma(g, false, st); }};
      op.join = join;
      ops().push_back(op);
      return;
    }
    tc->emplace_back();
    TcGemmLaunch& L = tc->back();
    L.w = &pc.tc;
    TcGemmParams& p = L.p;
    memset(&p, 0, sizeof(p));
    p.mode = e->cfg.gemm_mode;
    p.is3x3 = 0;
    p.bf16_in = bf ? 1 : 0;
    p.out_bf16 = out.es == 2 ? 1 : 0;
    if (bf && pass) { error = "bf16 mode: the pass-through GEMM epilogue is not built (unit tails go through dwpw): " + name; return; }
    p.num_steps = pc.tc.Kpad / (bf ? 64 : kTcBK);
    p.chunks_per_tap = p.num_steps;
    p.ksub = bf ? (pc.ktot + 15) / 16 : (pc.ktot + 7) / 8;      // valid 32-byte K sub-steps
    p.M = M;
    p.num_tiles = (M + kTcBM - 1) / kTcBM;
    p.N = pc.n; p.Npad = pc.tc.Npad;
    // head_det_*.4 (K = 96, N = 255): single merged accumulator, in the raw tail too so that the
    // raw-map parity tests measure exactly the sums the fused decode epilogue consumes
    tc_plan_tmem(p, name.size() > 2 && name.compare(0, 8, "head_det") == 0 && name.compare(name.size() - 2, 2, ".4") == 0);
    p.a_box_bytes = kTcAStageBytes;
    p.out = out.p; p.out_ld = out.ld; p.out_off = out_off; p.out_step = out_step;
    p.bias = pc.b_dev; p.act = c.act;
    p.pass = pass ? pass->p : nullptr; p.pass_ld = pass ? pass->ld : 0;
    p.err_flag = e->d_err;
    if (dec) {
      p.dec = *dec;
      L.dec_classes = e->cfg.num_classes;
    }
    const int oal = 16 / out.es;                                // output elements per 16 bytes
    p.tma_store = (!dec && !pass && out_step == 1 && out_off % oal == 0 && out.ld % oal == 0) ? 1 : 0;
    if (p.tma_store && !make_tmap_out(&L.tmOut, out.at(out_off), (uint64_t)round_up(pc.n, oal), (uint64_t)M,
                                      (uint64_t)out.ld, out.es == 2)) {
      error = "cuTensorMapEncodeTiled failed for output of " + name;
      return;
    }
    if (!make_tmap_2d(&L.tmA, in.at(in_off), (uint64_t)pc.ktot, (uint64_t)M, (uint64_t)in.ld, kTcBM, bf)) {
      error = "cuTensorMapEncodeTiled failed for input of " + name;
      return;
    }
    if (!tc_plan_smem(L)) { error = "no smem configuration for " + name; return; }
    L.grid = (unsigned)std::min<int64_t>(p.num_tiles, kNumSMs);
    const TcGemmLaunch* Lp = &L;
    // fused decode: the raw map (4*M*cout) is not written; boxes/scores/classes (24 B per anchor) are
    const double obytes = dec ? abytes - (double)out.es * M * c.cout + 24.0 * M * 3 : abytes;
    Op op{dec ? name + "+decode" : name, dec ? "pw_decode_tcgen05" : "pw_tcgen05", obytes, aflops,
          [=](cudaStream_t st) { return launch_tc_gemm(*Lp, st); }};
    op.join = join;
    ops().push_back(op);
  }

  // The two output convs of a stride-2 unit as one GEMM over K = [b1dw | mid2] (pack_cat): plain dense output.
  // Returns false when the unit keeps its two strided-store GEMMs (FFMA cross-check mode).
  bool catpw(int si, const std::string& unit, const Tensor& b1dw, const Tensor& mid2, const Tensor& out) {
    if (e->cfg.gemm_mode == YNB_GEMM_FP32_FFMA || e->cat[si].empty()) return false;
    const bool bf = is_bf16(e);
    const int64_t M = (int64_t)B * out.H * out.W;
    const ConvSpec& c1 = spec(unit + "branch1.2");
    const ConvSpec& c2 = spec(unit + "branch2.5");
    for (size_t pi = 0; pi < e->cat[si].size(); ++pi) {
      const ynb_engine::CatConv& cc = e->cat[si][pi];
      tc->emplace_back();
      TcGemmLaunch& L = tc->back();
      L.w = &cc.pc.tc;
      TcGemmParams& p = L.p;
      memset(&p, 0, sizeof(p));
      p.mode = e->cfg.gemm_mode;
      p.bf16_in = bf ? 1 : 0;
      p.out_bf16 = out.es == 2 ? 1 : 0;
      const int ch = bf ? 64 : kTcBK;
      p.num_steps = cc.pc.tc.Kpad / ch;
      p.chunks_per_tap = p.num_steps;
      p.a2_step = cc.k1p / ch;
      p.ksub = 0;                                   // both K blocks are whole chunks (zero padded)
      p.M = M;
      p.num_tiles = (M + kTcBM - 1) / kTcBM;
      p.N = cc.pc.n; p.Npad = cc.pc.tc.Npad;
      tc_plan_tmem(p);
      p.a_box_bytes = kTcAStageBytes;
      p.out = out.p; p.out_ld = out.ld; p.out_off = cc.n0; p.out_step = 1;
      p.bias = cc.pc.b_dev; p.act = c1.act;
      p.err_flag = e->d_err;
      p.tma_store = 1;
      const int oal = 16 / out.es;
      if (!make_tmap_out(&L.tmOut, out.at(cc.n0), (uint64_t)round_up(cc.pc.n, oal), (uint64_t)M, (uint64_t)out.ld, out.es == 2) ||
          !make_tmap_2d(&L.tmA, b1dw.p, (uint64_t)b1dw.ld, (uint64_t)M, (uint64_t)b1dw.ld, kTcBM, bf) ||
          !make_tmap_2d(&L.tmAlo, mid2.p, (uint64_t)mid2.ld, (uint64_t)M, (uint64_t)mid2.ld, kTcBM, bf)) {
        error = "cuTensorMapEncodeTiled failed for the merged stride-2 conv of " + unit;
        return true;
      }
      if (!tc_plan_smem(L)) { error = "no smem configuration for the merged stride-2 conv of " + unit; return true; }
      L.grid = (unsigned)std::min<int64_t>(p.num_tiles, kNumSMs);
      const TcGemmLaunch* Lp = &L;
      const double frac = (double)cc.pc.n / out.ld;
      const double bytes = (double)b1dw.es * M * (c1.cin + c2.cin) + (double)out.es * M * 2.0 * c1.cout * frac +
                           (bf ? 2.0 : 4.0) * (c1.cin + c2.cin) * c1.cout;
      const double flops = 2.0 * M * (c1.cin + c2.cin) * c1.cout * frac;
      ops().push_back({unit + "branch1.2|branch2.5" + (e->cat[si].size() > 1 ? "." + std::to_string(pi) : ""), "pw_tcgen05", bytes,
                       flops, [=](cudaStream_t st) { return launch_tc_gemm(*Lp, st); }});
    }
    return true;
  }

  // Fused depthwise 3x3 (stride 1) -> pointwise conv in ONE launch (unit_tc.cuh); `pass` as in pw().
  // Returns false when the pair has to stay unfused (FFMA cross-check mode, shape does not fit).
  bool dwpw(const std::string& dw_name, const std::string& pw_name, const Tensor& in, const Tensor& out,
            const Tensor* pass) {
    if (e->cfg.gemm_mode == YNB_GEMM_FP32_FFMA) return false;
    const PackedConv& dc = conv(dw_name);
    const PackedConv& pc = conv(pw_name);
    const ConvSpec& ds = spec(dw_name);
    const ConvSpec& ps = spec(pw_name);
    if (ds.stride != 1 || dc.n != pc.ktot) return false;
    dp->emplace_back();
    DwPwLaunch& L = dp->back();
    DwPwParams& p = L.p;
    memset(&p, 0, sizeof(p));
    p.dw_w = dc.w_dev; p.dw_b = dc.b_dev; p.dw_act = ds.act;
    p.out = out.p; p.out_ld = out.ld; p.out_off = 0;
    p.bias = pc.b_dev; p.act = ps.act;
    p.pass = pass ? pass->p : nullptr; p.pass_ld = pass ? pass->ld : 0;
    p.err_flag = e->d_err;
    if (!plan_dwpw(L, in.p, in.ld, B, in.H, in.W, ds.cin, dc.n, &pc.tc, e->cfg.gemm_mode)) {
      dp->pop_back();
      return false;
    }
    const double M = (double)B * in.H * in.W;
    const double bytes = (double)in.es * M * (ds.cin + ps.cout * (pass ? 3.0 : 1.0)) + (double)in.es * ps.cin * ps.cout +
                         4.0 * ps.cout + 40.0 * ds.cin;
    const double flops = 2.0 * M * ps.cin * ps.cout + 18.0 * M * ds.cin;
    const DwPwLaunch* Lp = &L;
    ops().push_back({dw_name + "+pw", "dwpw_tcgen05", bytes, flops,
                     [=](cudaStream_t st) { return launch_dwpw_tc(*Lp, st); }});
    return true;
  }

  // dense 3x3 (smooth): out = act(conv3x3(a + resample(a2)))
  void conv3(const std::string& name, const Tensor& a, const Tensor* a2, int a2_mode, const Tensor& sum,
             const Tensor& sum_lo, const Tensor& out) {
    const PackedConv& pc = conv(name);
    const ConvSpec& c = spec(name);
    int64_t M = (int64_t)B * a.H * a.W;
    const bool bf = is_bf16(e);
    const double eb = a.es;
    const double wbytes = eb * 9 * c.cin * c.cout + 4.0 * c.cout;
    const double aflops = 2.0 * M * 9 * c.cin * c.cout;
    // fused form reads a and the useful part of a2 once and writes the output once
    const double a2bytes = a2 ? eb * c.cin * M * (a2_mode == 1 ? 0.25 : 1.0) : 0.0;
    if (e->cfg.gemm_mode == YNB_GEMM_FP32_FFMA) {
      GemmParams g{};
      g.a = a.p; g.a_ld = a.ld; g.a_off = 0;
      g.a2 = a2 ? a2->p : nullptr; g.a2_ld = a2 ? a2->ld : 0; g.a2_mode = a2 ? a2_mode : 0;
      g.H = a.H; g.W = a.W; g.C = c.cin;
      g.w = pc.w_dev; g.bias = pc.b_dev; g.out = out.p; g.out_ld = out.ld; g.out_off = 0; g.out_step = 1;
      g.M = M; g.N = pc.n; g.Ktot = pc.ktot; g.act = c.act;
      plan->net.push_back({name, "conv3x3_ffma", 4.0 * M * (c.cin + c.cout) + a2bytes + wbytes, aflops,
                           [=](cudaStream_t st) { return launch_gemm_ffma(g, true, st); }});
      return;
    }
    // tensor-core path: materialise the sum once (HBM-bound elementwise), then 9 shifted TMA boxes
    Tensor src = a;
    // fp32-parity mode: the merge kernel writes the sum as exact-tf32 hi + lo planes once, instead of the
    // GEMM splitting every element nine times (once per tap)
    const bool presplit = a2 != nullptr && e->cfg.gemm_mode == YNB_GEMM_TC_3XTF32;
    if (a2) {
      Tensor a_ = a, a2_ = *a2, s_ = sum, sl_ = sum_lo;
      int B_ = B;
      plan->net.push_back({name + "+merge", "resample_add", (presplit ? 3.0 : 2.0) * eb * M * c.cin + a2bytes,
                           1.0 * M * c.cin, [=](cudaStream_t st) {
        return launch_resample_add(a_.p, a2_.p, s_.p, presplit ? sl_.p : nullptr, B_, a_.H, a_.W, a_.ld, a2_mode, st, bf);
      }});
      src = sum;
    }
    tc->emplace_back();
    TcGemmLaunch& L = tc->back();
    L.w = &pc.tc;
    TcGemmParams& p = L.p;
    memset(&p, 0, sizeof(p));
    p.mode = e->cfg.gemm_mode;
    p.is3x3 = 1;
    p.bf16_in = bf ? 1 : 0;
    p.out_bf16 = out.es == 2 ? 1 : 0;
    p.chunks_per_tap = bf ? (c.cin + 63) / 64 : c.cin / kTcBK;   // bf16: every tap padded to whole 64-channel chunks
    p.num_steps = 9 * p.chunks_per_tap;
    p.H = a.H; p.W = a.W;
    tc_pick_tile(p.H, p.W, &p.TH, &p.TW);
    p.tiles_x = (p.W + p.TW - 1) / p.TW;
    p.tiles_y = (p.H + p.TH - 1) / p.TH;
    p.num_tiles = (int64_t)B * p.tiles_x * p.tiles_y;
    p.M = M;
    p.N = pc.n; p.Npad = pc.tc.Npad;
    tc_plan_tmem(p);
    p.a_box_bytes = (uint32_t)(p.TH * p.TW * 128);
    p.out = out.p; p.out_ld = out.ld; p.out_off = 0; p.out_step = 1;
    p.bias = pc.b_dev; p.act = c.act;
    p.err_flag = e->d_err;
    if (!make_tmap_nhwc(&L.tmA, src.p, c.cin, src.W, src.H, B, src.ld, p.TW, p.TH, bf) ||
        (presplit && !make_tmap_nhwc(&L.tmAlo, sum_lo.p, c.cin, src.W, src.H, B, src.ld, p.TW, p.TH))) {
      error = "cuTensorMapEncodeTiled failed for input of " + name;
      return;
    }
    p.presplit = presplit ? 1 : 0;
    if (!tc_plan_smem(L)) { error = "no smem configuration for " + name; return; }
    L.grid = (unsigned)std::min<int64_t>(p.num_tiles, kNumSMs);
    const TcGemmLaunch* Lp = &L;
    plan->net.push_back({name, "conv3x3_tcgen05", eb * M * (c.cin + c.cout) + wbytes, aflops,
                         [=](cudaStream_t st) { return launch_tc_gemm(*Lp, st); }});
  }
};

int build_plan(ynb_engine* e, int B, Plan** out) {
  auto it = e->plans.find(B);
  if (it != e->plans.end()) { *out = it->second.get(); return YNB_OK; }
  auto plan = std::make_unique<Plan>();
  plan->batch = B;
  e->tc_store.emplace_back();
  e->dp_store.emplace_back();
  Planner P{e, B, plan.get(), &e->tc_store.back(), &e->dp_store.back(), ""};
  const int S = e->S;

  // stem + pool
  {
    Tensor pool = P.T("pool");
    // input pointer is bound at run time (first op takes it from the engine)
    double px = (double)B * S * S;
    const bool bf = is_bf16(e);
    plan->net.push_back({"backbone.conv1.0+maxpool", "stem_pool", 4.0 * 3 * px + (bf ? 2.0 : 4.0) * 24 * px / 16 + 4.0 * 27 * 24,
                         2.0 * 27 * 24 * px / 4, [=](cudaStream_t st) {
      // the input pointer is the caller's: one tensor map per (pointer, batch, S), built on first sight
      const float* xin = e->d_x_bound;
      auto key = std::make_tuple(xin, B, S);   // the map encodes dims / strides from S
      auto it = e->stem_maps.find(key);
      if (it == e->stem_maps.end()) {
        ynb_engine::StemMap sm{};
        sm.ok = make_tmap_stem_input(&sm.tm, xin, S, B) ? 1 : 0;
        if (e->stem_maps.size() > 64) e->stem_maps.clear();
        it = e->stem_maps.emplace(key, sm).first;
      }
      return launch_stem_pool(xin, pool.p, bf, e->stem_w, it->second.tm, it->second.ok, B, S, st);
    }});
  }
  Tensor x = P.T("pool");
  for (int si = 0; si < 3; ++si) {
    std::string st = "stage" + std::to_string(si + 2);
    std::string bk = "backbone." + st + ".";
    int h = stage_channels()[si + 1] / 2;
    Tensor b1dw = P.T(st + ".b1dw"), b2pw = P.T(st + ".b2pw"), mid1 = P.T(st + ".mid1"), mid2 = P.T(st + ".mid2");
    // ---- stride-2 unit: out[2i] = branch1, out[2i+1] = branch2 (shufflenetv2.py:73-76)
    Tensor o0 = P.T(st + ".0");
    P.dw(bk + "0.branch1.0", x, 0, b1dw);
    if (si > 0) plan->net.back().join = true;    // x = previous stage's last unit (side copy pending)
    P.pw(bk + "0.branch2.0", x, 0, b2pw, 0, 1);
    P.dw(bk + "0.branch2.3", b2pw, 0, mid2);
    if (!P.catpw(si, bk + "0.", b1dw, mid2, o0)) {
      P.pw(bk + "0.branch1.2", b1dw, 0, o0, 0, 2);
      P.pw(bk + "0.branch2.5", mid2, 0, o0, 1, 2);
    }
    x = o0;
    // ---- stride-1 units: x1 passes through to slot 2i, branch2(x2) lands in slot 2i+1 (:70-76)
    for (int bi = 1; bi < stage_repeats()[si]; ++bi) {
      std::string u = bk + std::to_string(bi);
      Tensor o = P.T(st + "." + std::to_string(bi));
      const int x2_off = x2_window(h, is_bf16(e) ? 8 : 4).off;
      // the previous unit's pass-through copy wrote half of x: join before reading it
      const bool ffma = e->cfg.gemm_mode == YNB_GEMM_FP32_FFMA;
      P.pw(u + ".branch2.0", x, x2_off, mid1, 0, 1, /*join=*/ffma && bi > 1);
      if (ffma) {   // cross-check path: pass-through as a side-stream copy next to the unit's convs
        plan->net.back().mark = true;            // fork point: x is complete here
        P.passthrough(u, x, o, h);               // o[2i] = x[i]
      }
      // tensor-core path: depthwise + pointwise fused, the epilogue writes whole interleaved rows (x1 | branch2)
      if (!P.dwpw(u + ".branch2.3", u + ".branch2.5", mid1, o, &x)) {
        P.dw(u + ".branch2.3", mid1, 0, mid2);
        P.pw(u + ".branch2.5", mid2, 0, o, 1, 2, false, &x);
      }
      x = o;
    }
  }
  // ---- neck (models/yolo_nano.py:286-296)
  Tensor c3 = P.T("c3"), c4 = P.T("c4"), c5 = P.T("c5");
  Tensor lat3 = P.T("lat3"), lat4 = P.T("lat4"), lat5 = P.T("lat5");
  P.pw("conv1x1_0.convs.0", c3, 0, lat3, 0, 1, /*join=*/true);   // c5's pass-through copy may be in flight
  P.pw("conv1x1_1.convs.0", c4, 0, lat4, 0, 1);
  P.pw("conv1x1_2.convs.0", c5, 0, lat5, 0, 1);
  Tensor fpn4 = P.T("fpn4"), p3 = P.T("p3"), p4 = P.T("p4"), p5 = P.T("p5");
  P.conv3("smooth_0.convs.0", lat4, &lat5, 1, P.T("sum4"), P.T("sum4.lo"), fpn4);
  P.conv3("smooth_1.convs.0", lat3, &fpn4, 1, P.T("sum3"), P.T("sum3.lo"), p3);
  P.conv3("smooth_2.convs.0", fpn4, &p3, 2, P.T("sum4b"), P.T("sum4b.lo"), p4);
  P.conv3("smooth_3.convs.0", lat5, &p4, 2, P.T("sum5"), P.T("sum5.lo"), p5);
  // ---- heads (models/yolo_nano.py:50-70, 299-301)
  Tensor feats[3] = {p3, p4, p5};
  Tensor head_in[3];
  for (int l = 0; l < 3; ++l) {
    std::string hd = "head_det_" + std::to_string(l + 1);
    Tensor ta = P.T("head" + std::to_string(l) + ".a"), tb = P.T("head" + std::to_string(l) + ".b");
    if (!P.dwpw(hd + ".0.convs.0", hd + ".1.convs.0", feats[l], ta, nullptr)) {
      P.dw(hd + ".0.convs.0", feats[l], 0, tb);
      P.pw(hd + ".1.convs.0", tb, 0, ta, 0, 1);
    }
    if (!P.dwpw(hd + ".2.convs.0", hd + ".3.convs.0", ta, tb, nullptr)) {
      Tensor tc2 = P.T("head" + std::to_string(l) + ".c");
      P.dw(hd + ".2.convs.0", ta, 0, tc2);
      P.pw(hd + ".3.convs.0", tc2, 0, tb, 0, 1);
    }
    head_in[l] = tb;
  }
  P.dst = &plan->raw_tail;
  for (int l = 0; l < 3; ++l) P.pw("head_det_" + std::to_string(l + 1) + ".4", head_in[l], 0, e->raw[l], 0, 1);
  // fused tail: tensor-core modes with the class counts the decode epilogue is instantiated for
  plan->fused = e->cfg.gemm_mode != YNB_GEMM_FP32_FFMA && e->cfg.num_anchors == 3 &&
                (e->cfg.num_classes == 80 || e->cfg.num_classes == 20);
  if (plan->fused) {
    P.dst = &plan->fused_tail;
    int64_t off = 0;
    for (int l = 0; l < 3; ++l) {
      TcGemmParams::Decode d{};
      const int stride = 8 << l;
      d.boxes = e->d_boxes; d.scores = e->d_scores; d.cls = e->d_cls;
      d.G = S / stride; d.HW = d.G * d.G;
      d.stride = (float)stride; d.input_size = (float)S;
      for (int a = 0; a < 3; ++a) {
        d.aw[a] = e->cfg.anchors[(l * 3 + a) * 2];
        d.ah[a] = e->cfg.anchors[(l * 3 + a) * 2 + 1];
      }
      d.Ntot = e->N(); d.level_off = off;
      off += (int64_t)d.HW * 3;
      P.pw("head_det_" + std::to_string(l + 1) + ".4", head_in[l], 0, e->raw[l], 0, 1, false, nullptr, &d);
    }
  }
  P.dst = nullptr;
  if (!P.error.empty()) return fail(e, YNB_ERR_CUDA, P.error);
  // ---- decode (models/yolo_nano.py:303-330, 362-367)
  int64_t N = e->N(), off = 0;
  for (int l = 0; l < 3; ++l) {
    DecodeParams d{};
    int stride = 8 << l;
    d.raw = e->raw[l].p; d.ld = e->raw[l].ld;
    d.boxes = e->d_boxes; d.scores = e->d_scores; d.cls = e->d_cls;
    d.batch = B; d.G = S / stride; d.A = e->cfg.num_anchors; d.C = e->cfg.num_classes;
    d.stride = (float)stride; d.input_size = (float)S;
    for (int a = 0; a < d.A; ++a) {
      d.anchor_w[a] = e->cfg.anchors[(l * d.A + a) * 2];
      d.anchor_h[a] = e->cfg.anchors[(l * d.A + a) * 2 + 1];
    }
    d.N = N; d.level_off = off;
    off += (int64_t)d.G * d.G * d.A;
    double cells = (double)B * d.G * d.G;
    plan->decode.push_back({"decode.level" + std::to_string(l), "decode",
                            4.0 * cells * d.A * (1 + d.C + 4) + 24.0 * cells * d.A, 0.0,
                            [=](cudaStream_t st) { return launch_decode_level(d, st); }});
  }
  *out = plan.get();
  e->plans[B] = std::move(plan);
  return YNB_OK;
}

int check_ready(ynb_engine* e, int batch) {
  if (!e) return YNB_ERR_INVALID;
  if (!e->committed) return fail(e, YNB_ERR_STATE, "weights not committed (ynb_load_conv x77, ynb_commit_weights)");
  if (batch <= 0) return fail(e, YNB_ERR_INVALID, "batch must be positive");
  return YNB_OK;
}

cudaEvent_t next_event(ynb_engine* e) {
  cudaEvent_t ev = e->events[e->ev_next];
  e->ev_next = (e->ev_next + 1) % e->events.size();
  return ev;
}

// Runs a list of launches on the engine streams: main stream in order, `side` ops forked
// after the latest `mark` and joined where an op asks for it (and at the end).  Works the
// same eagerly and under stream capture (the fork/join events become graph edges).
struct SideState {
  cudaEvent_t mark = nullptr, done = nullptr;
};

int run_ops(ynb_engine* e, const std::vector<Op>& ops, SideState* ss = nullptr) {
  cudaStream_t st = e->s_main;
  SideState local;
  if (!ss) ss = &local;
  if (!e->profiling) {
    for (const Op& op : ops) {
      if (op.mark) {
        ss->mark = next_event(e);
        CUDA_TRY(e, cudaEventRecord(ss->mark, st));
      }
      if (op.join && ss->done) {
        CUDA_TRY(e, cudaStreamWaitEvent(st, ss->done, 0));
        ss->done = nullptr;
      }
      cudaError_t r;
      if (op.side) {
        if (!ss->mark) {
          ss->mark = next_event(e);
          CUDA_TRY(e, cudaEventRecord(ss->mark, st));
        }
        CUDA_TRY(e, cudaStreamWaitEvent(e->s_side, ss->mark, 0));
        r = op.fn(e->s_side);
        ss->done = next_event(e);
        CUDA_TRY(e, cudaEventRecord(ss->done, e->s_side));
      } else {
        r = op.fn(st);
      }
      if (r != cudaSuccess)
        return fail(e, YNB_ERR_CUDA, "kernel launch (" + op.name + "): " + cudaGetErrorString(r));
    }
    if (ss == &local && ss->done) CUDA_TRY(e, cudaStreamWaitEvent(st, ss->done, 0));
    return YNB_OK;
  }
  // profiling pass: everything serialised on the main stream, one CUDA event pair per launch
  std::vector<cudaEvent_t> ev(ops.size() + 1);
  for (auto& x : ev) CUDA_TRY(e, cudaEventCreate(&x));
  CUDA_TRY(e, cudaEventRecord(ev[0], st));
  for (size_t i = 0; i < ops.size(); ++i) {
    cudaError_t r = ops[i].fn(st);
    if (r != cudaSuccess)
      return fail(e, YNB_ERR_CUDA, "kernel launch (" + ops[i].name + "): " + cudaGetErrorString(r));
    CUDA_TRY(e, cudaEventRecord(ev[i + 1], st));
  }
  CUDA_TRY(e, cudaEventSynchronize(ev.back()));
  for (size_t i = 0; i < ops.size(); ++i) {
    float ms = 0;
    CUDA_TRY(e, cudaEventElapsedTime(&ms, ev[i], ev[i + 1]));
    e->prof.push_back({ops[i].name, ops[i].kind, ops[i].bytes, ops[i].flops, ms});
  }
  for (auto& x : ev) cudaEventDestroy(x);
  return YNB_OK;
}

// Orders the engine's main stream after the caller's stream ...
int enter(ynb_engine* e, cudaStream_t user) {
  CUDA_TRY(e, cudaEventRecord(e->ev_in, user));
  CUDA_TRY(e, cudaStreamWaitEvent(e->s_main, e->ev_in, 0));
  return YNB_OK;
}
// ... and the caller's stream after the engine's work.
int leave(ynb_engine* e, cudaStream_t user) {
  CUDA_TRY(e, cudaEventRecord(e->ev_out, e->s_main));
  CUDA_TRY(e, cudaStreamWaitEvent(user, e->ev_out, 0));
  return YNB_OK;
}

// Prepares workspace + plan for `batch` (may allocate: never called under capture).
int prepare(ynb_engine* e, int batch, Plan** plan_out) {
  int rc = check_ready(e, batch);
  if (rc) return rc;
  CUDA_TRY(e, cudaSetDevice(e->cfg.device));
  if ((rc = ensure_workspace(e, batch))) return rc;
  return build_plan(e, batch, plan_out);
}

// backbone + neck + heads on the engine's main stream
// stem .. raw head maps (the parity hook's path)
int run_network(ynb_engine* e, const float* x_dev, Plan* plan) {
  e->d_x_bound = x_dev;
  e->prof.clear();
  int rc = run_ops(e, plan->net);
  return rc ? rc : run_ops(e, plan->raw_tail);
}

// stem .. decoded boxes / scores / classes in the engine buffers (the product path)
int run_decoded(ynb_engine* e, const float* x_dev, Plan* plan) {
  if (!plan->fused) {
    int rc = run_network(e, x_dev, plan);
    return rc ? rc : run_ops(e, plan->decode);
  }
  e->d_x_bound = x_dev;
  e->prof.clear();
  int rc = run_ops(e, plan->net);
  return rc ? rc : run_ops(e, plan->fused_tail);
}

int check_device_error(ynb_engine* e) {
  cudaStream_t st = e->s_main;
  int flag = 0;
  CUDA_TRY(e, cudaMemcpyAsync(&flag, e->d_err, 4, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(e, cudaStreamSynchronize(st));
  if (flag != 0) {
    cudaMemsetAsync(e->d_err, 0, 4, st);
    return fail(e, YNB_ERR_CUDA, "tensor-core pipeline timed out waiting on mbarrier (code " +
                                     std::to_string(flag) + ")");
  }
  return YNB_OK;
}

}  // namespace

static void drop_graphs(ynb_engine* e);

// =============================================================================================
// C ABI
// =============================================================================================
YNB_EXPORT int ynb_abi_version(void) { return YNB_ABI_VERSION; }

YNB_EXPORT const char* ynb_last_error(const ynb_engine* e) { return e ? e->err.c_str() : g_create_error.c_str(); }

YNB_EXPORT int ynb_create(const ynb_config* cfg, ynb_engine** out) {
  if (!cfg || !out) return fail(nullptr, YNB_ERR_INVALID, "null argument");
  *out = nullptr;
  if (cfg->abi_version != YNB_ABI_VERSION) return fail(nullptr, YNB_ERR_INVALID, "ABI version mismatch");
  if (cfg->num_anchors != 3) return fail(nullptr, YNB_ERR_UNSUPPORTED, "num_anchors must be 3");
  if (cfg->num_classes < 1 || cfg->num_classes > 255) return fail(nullptr, YNB_ERR_INVALID, "num_classes out of range");
  if (cfg->input_size < 32 || cfg->input_size % 32 || cfg->input_size > 1024)
    return fail(nullptr, YNB_ERR_INVALID, "input_size must be a multiple of 32 in [32, 1024]");
  if (cfg->gemm_mode < 0 || cfg->gemm_mode > YNB_GEMM_TC_BF16) return fail(nullptr, YNB_ERR_INVALID, "bad gemm_mode");
  int ndev = 0;
  cudaError_t st = cudaGetDeviceCount(&ndev);
  if (st != cudaSuccess || ndev == 0)
    return fail(nullptr, YNB_ERR_NO_DEVICE,
                std::string("no CUDA device: ") + (st != cudaSuccess ? cudaGetErrorString(st) : "count is 0") +
                    " (this library has no CPU path)");
  if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, YNB_ERR_INVALID, "device ordinal out of range");
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, cfg->device) != cudaSuccess || prop.major != 10)
    return fail(nullptr, YNB_ERR_NO_DEVICE, "device is not compute capability 10.x (built for sm_100a only)");
  if (cudaSetDevice(cfg->device) != cudaSuccess) return fail(nullptr, YNB_ERR_CUDA, "cudaSetDevice failed");
  ynb_engine* e = new ynb_engine();
  e->cfg = *cfg;
  if (e->cfg.max_batch < 1) e->cfg.max_batch = 1;
  e->S = cfg->input_size;
  {   // ValTransforms defaults (data/transforms.py:447), BGR order
    const float mean[3] = {0.406f, 0.456f, 0.485f}, stdv[3] = {0.225f, 0.224f, 0.229f};
    make_prelut(&e->prelut, mean, stdv);
  }
  e->table = conv_table(cfg->num_classes, cfg->num_anchors);
  e->convs.resize(e->table.size());
  for (size_t i = 0; i < e->table.size(); ++i) e->index[e->table[i].name] = (int)i;
  bool ok = cudaStreamCreateWithFlags(&e->s_main, cudaStreamNonBlocking) == cudaSuccess &&
            cudaStreamCreateWithFlags(&e->s_side, cudaStreamNonBlocking) == cudaSuccess &&
            cudaEventCreateWithFlags(&e->ev_in, cudaEventDisableTiming) == cudaSuccess &&
            cudaEventCreateWithFlags(&e->ev_out, cudaEventDisableTiming) == cudaSuccess;
  ok = ok && cudaStreamCreateWithFlags(&e->s_copy, cudaStreamNonBlocking) == cudaSuccess;
  ok = ok && cudaStreamCreateWithFlags(&e->s_copy2, cudaStreamNonBlocking) == cudaSuccess;
  ok = ok && cudaEventCreateWithFlags(&e->ev_copy2, cudaEventDisableTiming) == cudaSuccess;
  ok = ok && cudaStreamCreateWithFlags(&e->s_d2h, cudaStreamNonBlocking) == cudaSuccess;
  ok = ok && cudaMalloc(&e->d_prelut, sizeof(PreLut)) == cudaSuccess &&
       cudaMemcpy(e->d_prelut, &e->prelut, sizeof(PreLut), cudaMemcpyHostToDevice) == cudaSuccess;
  for (int k = 0; k < 2 && ok; ++k)
    ok = cudaEventCreateWithFlags(&e->slot[k].h2d, cudaEventDisableTiming) == cudaSuccess &&
         cudaEventCreateWithFlags(&e->slot[k].done, cudaEventDisableTiming) == cudaSuccess &&
         cudaHostAlloc(&e->slot[k].flag_host, 64, cudaHostAllocDefault) == cudaSuccess;
  e->events.resize(64);
  for (auto& ev : e->events) ok = ok && cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) == cudaSuccess;
  if (!ok) {
    delete e;
    return fail(nullptr, YNB_ERR_CUDA, "stream / event creation failed");
  }
  *out = e;
  return YNB_OK;
}

static void drop_graphs(ynb_engine* e) {
  for (auto& kv : e->graphs) cudaGraphExecDestroy(kv.second);
  e->graphs.clear();
  e->graph_seen.clear();
}

YNB_EXPORT void ynb_destroy(ynb_engine* e) {
  if (!e) return;
  cudaSetDevice(e->cfg.device);
  cudaDeviceSynchronize();
  drop_graphs(e);
  for (auto ev : e->events) cudaEventDestroy(ev);
  if (e->ev_in) cudaEventDestroy(e->ev_in);
  if (e->ev_out) cudaEventDestroy(e->ev_out);
  for (int k = 0; k < 2; ++k) {
    if (e->slot[k].h2d) cudaEventDestroy(e->slot[k].h2d);
    if (e->slot[k].done) cudaEventDestroy(e->slot[k].done);
    if (e->slot[k].flag_host) cudaFreeHost(e->slot[k].flag_host);
  }
  if (e->s_copy) cudaStreamDestroy(e->s_copy);
  if (e->s_copy2) cudaStreamDestroy(e->s_copy2);
  if (e->ev_copy2) cudaEventDestroy(e->ev_copy2);
  if (e->s_d2h) cudaStreamDestroy(e->s_d2h);
  if (e->d_prelut) cudaFree(e->d_prelut);
  if (e->s_main) cudaStreamDestroy(e->s_main);
  if (e->s_side) cudaStreamDestroy(e->s_side);
  for (PackedConv& pc : e->convs) {
    if (pc.w_dev) cudaFree(pc.w_dev);
    if (pc.b_dev) cudaFree(pc.b_dev);
    if (pc.tc.hi) cudaFree(pc.tc.hi);
    if (pc.tc.lo) cudaFree(pc.tc.lo);
    if (pc.tc.bw) cudaFree(pc.tc.bw);
  }
  for (int si = 0; si < 3; ++si)
    for (auto& cc : e->cat[si]) {
      if (cc.pc.b_dev) cudaFree(cc.pc.b_dev);
      if (cc.pc.tc.hi) cudaFree(cc.pc.tc.hi);
      if (cc.pc.tc.lo) cudaFree(cc.pc.tc.lo);
      if (cc.pc.tc.bw) cudaFree(cc.pc.tc.bw);
    }
  if (e->ws) cudaFree(e->ws);
  delete e;
}

YNB_EXPORT int ynb_set_grid(ynb_engine* e, int32_t input_size) {
  if (!e) return YNB_ERR_INVALID;
  if (input_size < 32 || input_size % 32 || input_size > 1024)
    return fail(e, YNB_ERR_INVALID, "input_size must be a multiple of 32 in [32, 1024]");
  if (input_size != e->S) e->stem_maps.clear();
  e->S = input_size;   // workspace / plans are rebuilt lazily on the next forward
  return YNB_OK;
}

YNB_EXPORT int ynb_set_thresholds(ynb_engine* e, float conf, float nms, int32_t diou) {
  if (!e) return YNB_ERR_INVALID;
  e->cfg.conf_thresh = conf; e->cfg.nms_thresh = nms; e->cfg.diou_nms = diou;
  return YNB_OK;
}

YNB_EXPORT int ynb_set_gemm_mode(ynb_engine* e, int32_t mode) {
  if (!e) return YNB_ERR_INVALID;
  if (mode < 0 || mode > YNB_GEMM_TC_BF16) return fail(e, YNB_ERR_INVALID, "bad gemm_mode");
  if ((mode == YNB_GEMM_TC_BF16) != (e->cfg.gemm_mode == YNB_GEMM_TC_BF16))
    return fail(e, YNB_ERR_UNSUPPORTED, "bf16 mode changes the activation storage and the weight packing: create the "
                                        "engine with gemm_mode = YNB_GEMM_TC_BF16 instead of switching");
  if (mode != e->cfg.gemm_mode) {
    cudaDeviceSynchronize();
    e->cfg.gemm_mode = mode; e->plans.clear(); e->tc_store.clear(); e->dp_store.clear(); e->dw_maps.clear(); drop_graphs(e);
  }
  return YNB_OK;
}

YNB_EXPORT int64_t ynb_num_boxes(const ynb_engine* e) { return e ? e->N() : 0; }

YNB_EXPORT int64_t ynb_workspace_bytes(const ynb_engine* e, int32_t batch) {
  if (!e || batch < 1) return 0;
  ynb_engine tmp;
  tmp.cfg = e->cfg;
  return (int64_t)layout_workspace(&tmp, batch, e->S, nullptr);
}

YNB_EXPORT int32_t ynb_num_convs(void) { return 77; }

YNB_EXPORT const char* ynb_conv_name(int32_t i) {
  static const std::vector<ConvSpec> t = conv_table(80, 3);
  return (i >= 0 && i < (int)t.size()) ? t[i].name.c_str() : nullptr;
}

YNB_EXPORT int ynb_conv_shape(int32_t i, int32_t num_classes, int32_t num_anchors, int32_t* cout,
                              int32_t* cin_per_group, int32_t* ksize) {
  std::vector<ConvSpec> t = conv_table(num_classes, num_anchors);
  if (i < 0 || i >= (int)t.size() || !cout || !cin_per_group || !ksize) return YNB_ERR_INVALID;
  *cout = t[i].cout;
  *cin_per_group = t[i].kind == kDw3x3 ? 1 : t[i].cin;
  *ksize = t[i].kind == kPw1x1 ? 1 : 3;
  return YNB_OK;
}

YNB_EXPORT int ynb_load_conv(ynb_engine* e, const char* name, const float* w, int64_t w_elems, const float* b,
                             int64_t b_elems) {
  if (!e || !name || !w || !b) return fail(e, YNB_ERR_INVALID, "null argument");
  auto it = e->index.find(name);
  if (it == e->index.end()) return fail(e, YNB_ERR_INVALID, std::string("unknown conv ") + name);
  const ConvSpec& c = e->table[it->second];
  int64_t expect = (int64_t)c.cout * (c.kind == kDw3x3 ? 1 : c.cin) * (c.kind == kPw1x1 ? 1 : 9);
  if (w_elems != expect || b_elems != c.cout)
    return fail(e, YNB_ERR_INVALID, std::string("shape mismatch for ") + name);
  PackedConv& pc = e->convs[it->second];
  pc.w_host.assign(w, w + w_elems);
  pc.b_host.assign(b, b + b_elems);
  pc.loaded = true;
  e->committed = false;
  return YNB_OK;
}

YNB_EXPORT int ynb_commit_weights(ynb_engine* e) {
  if (!e) return YNB_ERR_INVALID;
  CUDA_TRY(e, cudaSetDevice(e->cfg.device));
  for (size_t i = 0; i < e->convs.size(); ++i)
    if (!e->convs[i].loaded) return fail(e, YNB_ERR_STATE, "conv not loaded: " + e->table[i].name);
  CUDA_TRY(e, cudaDeviceSynchronize());   // nothing in flight may still read the old buffers
  e->plans.clear();
  e->tc_store.clear(); e->dp_store.clear(); e->dw_maps.clear();
  drop_graphs(e);
  for (size_t i = 0; i < e->convs.size(); ++i) {
    int rc = pack_conv(e, (int)i);
    if (rc) return rc;
  }
  // The merged stride-2 weights depend only on the storage type, not on the GEMM mode: pack them in FFMA mode too,
  // or a later ynb_set_gemm_mode to a tensor-core mode would run the stride-2 units on the previous weights.
  for (int si = 0; si < 3; ++si) {
    int rc = pack_cat(e, si);
    if (rc) return rc;
  }
  e->committed = true;
  return YNB_OK;
}

YNB_EXPORT int ynb_forward_raw(ynb_engine* e, const float* x_dev, int32_t batch, float* ps, float* pm, float* pl,
                               void* stream) {
  if (!e || !x_dev || !ps || !pm || !pl) return fail(e, YNB_ERR_INVALID, "null argument");
  cudaStream_t user = (cudaStream_t)stream;
  CounterScope cs(e);
  Plan* plan = nullptr;
  int rc = prepare(e, batch, &plan);
  if (rc || (rc = enter(e, user)) || (rc = run_network(e, x_dev, plan))) return rc;
  float* outs[3] = {ps, pm, pl};
  for (int l = 0; l < 3; ++l) {
    const Tensor& t = e->raw[l];
    CUDA_TRY(e, launch_nhwc_to_nchw(t.p, t.ld, outs[l], batch, t.C, t.H * t.W, e->s_main, t.es == 2));
  }
  if ((rc = leave(e, user))) return rc;
  return e->cfg.gemm_mode == YNB_GEMM_FP32_FFMA ? YNB_OK : check_device_error(e);
}

YNB_EXPORT int ynb_forward_decode(ynb_engine* e, const float* x_dev, int32_t batch, float* boxes, float* scores,
                                  int32_t* cls, void* stream) {
  if (!e || !x_dev || !boxes || !scores || !cls) return fail(e, YNB_ERR_INVALID, "null argument");
  cudaStream_t user = (cudaStream_t)stream;
  CounterScope cs(e);
  Plan* plan = nullptr;
  int rc = prepare(e, batch, &plan);
  if (rc || (rc = enter(e, user)) || (rc = run_decoded(e, x_dev, plan))) return rc;
  int64_t n = e->N();
  cudaStream_t st = e->s_main;
  CUDA_TRY(e, cudaMemcpyAsync(boxes, e->d_boxes, (size_t)batch * n * 16, cudaMemcpyDeviceToDevice, st));
  CUDA_TRY(e, cudaMemcpyAsync(scores, e->d_scores, (size_t)batch * n * 4, cudaMemcpyDeviceToDevice, st));
  CUDA_TRY(e, cudaMemcpyAsync(cls, e->d_cls, (size_t)batch * n * 4, cudaMemcpyDeviceToDevice, st));
  if ((rc = leave(e, user))) return rc;
  return e->cfg.gemm_mode == YNB_GEMM_FP32_FFMA ? YNB_OK : check_device_error(e);
}

// network + decode + NMS on the engine's main stream (eager, or into a stream capture)
static int detect_ops(ynb_engine* e, Plan* plan, const float* x_dev, int batch, float* ob, float* os, int32_t* oc,
                      int32_t* on) {
  int rc = run_decoded(e, x_dev, plan);
  if (rc) return rc;
  const int64_t n = e->N();
  std::vector<Op> nms_ops(1);
  // product path: anchor-grid NMS (nms_grid.cuh); the sorted greedy NMS stays as the generic
  // kernel (ynb_nms) and for the inputs the grid NMS does not take
  if (e->cfg.num_anchors == 3 && n <= 65535 && e->S % 32 == 0) {
    GridNmsWorkspace gw = grid_nms_carve(e->d_nms_ws, batch, n);
    const int S = e->S;
    nms_ops[0] = {"nms(prep+build+resolve+compact)", "nms", 24.0 * batch * n * 2, 0.0, [=](cudaStream_t s2) {
      return launch_nms_grid(e->d_boxes, e->d_scores, e->d_cls, batch, S, e->cfg.num_classes, e->cfg.conf_thresh,
                             e->cfg.nms_thresh, e->cfg.diou_nms, ob, os, oc, on, nullptr, gw, s2);
    }};
    return run_ops(e, nms_ops);
  }
  NmsWorkspace w = nms_carve(e->d_nms_ws, batch, e->N());
  nms_ops[0] = {"nms(keys+sort+greedy+compact)", "nms", 24.0 * batch * n * 2, 0.0, [=](cudaStream_t s2) {
    return launch_nms(e->d_boxes, e->d_scores, e->d_cls, batch, n, e->cfg.num_classes, e->cfg.conf_thresh,
                      e->cfg.nms_thresh, e->cfg.diou_nms, ob, os, oc, on, nullptr, w, s2);
  }};
  return run_ops(e, nms_ops);
}

// The whole path for device-resident input.  Steady state = ONE cudaGraphLaunch: the ~90
// launches of a forward are captured (with the side-stream fork/joins) the second time the
// same (batch, buffers, thresholds) combination is seen, and replayed afterwards.
static int detect_device(ynb_engine* e, const float* x_dev, int batch, float* ob, float* os, int32_t* oc,
                         int32_t* on) {
  Plan* plan = nullptr;
  int rc = prepare(e, batch, &plan);
  if (rc) return rc;
  if (!e->use_graphs || e->profiling) return detect_ops(e, plan, x_dev, batch, ob, os, oc, on);
  ynb_engine::GraphKey key{batch, x_dev, ob, os, oc, on, e->cfg.conf_thresh, e->cfg.nms_thresh,
                           e->cfg.diou_nms, e->cfg.gemm_mode, e->S};
  auto it = e->graphs.find(key);
  if (it == e->graphs.end()) {
    if (e->graph_seen.size() > 256) e->graph_seen.clear();      // callers that never reuse a buffer stay eager
    if (e->graph_seen[key]++ == 0) return detect_ops(e, plan, x_dev, batch, ob, os, oc, on);   // first sighting
    if (e->graphs.size() >= 32) drop_graphs(e);
    cudaGraph_t graph = nullptr;
    CUDA_TRY(e, cudaStreamBeginCapture(e->s_main, cudaStreamCaptureModeThreadLocal));
    const int64_t l0 = e->counter.n;
    rc = detect_ops(e, plan, x_dev, batch, ob, os, oc, on);
    e->graph_launches[batch] = e->counter.n - l0;
    e->counter.n = l0;                       // captured, not launched
    cudaError_t ce = cudaStreamEndCapture(e->s_main, &graph);
    if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
    if (ce != cudaSuccess) return fail(e, YNB_ERR_CUDA, std::string("cudaStreamEndCapture: ") + cudaGetErrorString(ce));
    cudaGraphExec_t exec = nullptr;
    ce = cudaGraphInstantiate(&exec, graph, 0);
    cudaGraphDestroy(graph);
    if (ce != cudaSuccess) return fail(e, YNB_ERR_CUDA, std::string("cudaGraphInstantiate: ") + cudaGetErrorString(ce));
    it = e->graphs.emplace(key, exec).first;
  }
  CUDA_TRY(e, cudaGraphLaunch(it->second, e->s_main));
  e->counter.n += e->graph_launches[batch];
  return YNB_OK;
}

YNB_EXPORT int ynb_forward_detect(ynb_engine* e, const float* x_dev, int32_t batch, float* ob, float* os,
                                  int32_t* oc, int32_t* on, void* stream) {
  if (!e || !x_dev || !ob || !os || !oc || !on) return fail(e, YNB_ERR_INVALID, "null argument");
  cudaStream_t user = (cudaStream_t)stream;
  CounterScope cs(e);
  int rc = check_ready(e, batch);
  if (rc || (rc = enter(e, user)) || (rc = detect_device(e, x_dev, batch, ob, os, oc, on))) return rc;
  return leave(e, user);
}

// Host-buffer path, split in two so that consecutive steps overlap: submit(i+1) copies the
// next batch over PCIe on the copy stream while the compute stream is still busy with step i.
// x_host != nullptr: float32 [B,3,S,S] input; else img_host uint8 [B,S,S,3] BGR (+ optional rects)
static int submit_host_common(ynb_engine* e, int32_t slot_id, const float* x_host, const uint8_t* img_host,
                              const int32_t* rects_host, int32_t batch, float* ob, float* os, int32_t* oc,
                              int32_t* on, void* stream) {
  if (!e || (!x_host && !img_host) || !ob || !os || !oc || !on) return fail(e, YNB_ERR_INVALID, "null argument");
  if (slot_id < 0 || slot_id > 1) return fail(e, YNB_ERR_INVALID, "slot must be 0 or 1");
  cudaStream_t user = (cudaStream_t)stream;
  CounterScope cs(e);
  Plan* plan = nullptr;
  int rc = prepare(e, batch, &plan);
  if (rc) return rc;
  ynb_engine::HostSlot& sl = e->slot[slot_id];
  if (sl.busy) return fail(e, YNB_ERR_STATE, "slot still in flight: call ynb_wait_host first");
  const size_t px = (size_t)3 * e->S * e->S;
  // order after the caller's stream, then: H2D on the copy stream, compute on the main stream
  CUDA_TRY(e, cudaEventRecord(e->ev_in, user));
  CUDA_TRY(e, cudaStreamWaitEvent(e->s_copy, e->ev_in, 0));
  if (x_host) {
    // two halves on two copy streams (two DMA queues in flight)
    const size_t total = px * 4 * batch, half = (total / 2) & ~(size_t)255;
    CUDA_TRY(e, cudaStreamWaitEvent(e->s_copy2, e->ev_in, 0));
    CUDA_TRY(e, cudaMemcpyAsync(sl.x, x_host, half, cudaMemcpyHostToDevice, e->s_copy));
    CUDA_TRY(e, cudaMemcpyAsync(reinterpret_cast<char*>(sl.x) + half, reinterpret_cast<const char*>(x_host) + half,
                                total - half, cudaMemcpyHostToDevice, e->s_copy2));
    CUDA_TRY(e, cudaEventRecord(e->ev_copy2, e->s_copy2));
    CUDA_TRY(e, cudaStreamWaitEvent(e->s_copy, e->ev_copy2, 0));
  } else {
    CUDA_TRY(e, cudaMemcpyAsync(sl.img_u8, img_host, px * batch, cudaMemcpyHostToDevice, e->s_copy));
    if (rects_host)
      CUDA_TRY(e, cudaMemcpyAsync(sl.rects, rects_host, (size_t)batch * 16, cudaMemcpyHostToDevice, e->s_copy));
  }
  CUDA_TRY(e, cudaEventRecord(sl.h2d, e->s_copy));
  CUDA_TRY(e, cudaStreamWaitEvent(e->s_main, sl.h2d, 0));
  if (!x_host)   // uint8 HWC BGR -> normalised float32 NCHW RGB, 4x fewer bytes over PCIe
    CUDA_TRY(e, launch_preprocess_u8(sl.img_u8, rects_host ? sl.rects : nullptr, sl.x, e->d_prelut, batch, e->S,
                                     e->s_main));
  if ((rc = detect_device(e, sl.x, batch, sl.boxes, sl.scores, sl.cls, sl.counts))) return rc;
  CUDA_TRY(e, cudaMemcpyAsync(on, sl.counts, (size_t)batch * 4, cudaMemcpyDeviceToHost, e->s_main));
  CUDA_TRY(e, cudaMemcpyAsync(sl.flag_host, e->d_err, 4, cudaMemcpyDeviceToHost, e->s_main));
  CUDA_TRY(e, cudaEventRecord(sl.done, e->s_main));
  sl.busy = true; sl.batch = batch; sl.ob = ob; sl.os = os; sl.oc = oc; sl.on = on;
  return YNB_OK;
}

YNB_EXPORT int ynb_submit_host(ynb_engine* e, int32_t slot_id, const float* x_host, int32_t batch, float* ob,
                               float* os, int32_t* oc, int32_t* on, void* stream) {
  if (!x_host) return fail(e, YNB_ERR_INVALID, "null argument");
  return submit_host_common(e, slot_id, x_host, nullptr, nullptr, batch, ob, os, oc, on, stream);
}

YNB_EXPORT int ynb_submit_host_u8(ynb_engine* e, int32_t slot_id, const uint8_t* img_host, const int32_t* rects_host,
                                  int32_t batch, float* ob, float* os, int32_t* oc, int32_t* on, void* stream) {
  if (!img_host) return fail(e, YNB_ERR_INVALID, "null argument");
  return submit_host_common(e, slot_id, nullptr, img_host, rects_host, batch, ob, os, oc, on, stream);
}

YNB_EXPORT int ynb_set_normalization(ynb_engine* e, const float* mean_bgr, const float* std_bgr) {
  if (!e || !mean_bgr || !std_bgr) return fail(e, YNB_ERR_INVALID, "null argument");
  for (int c = 0; c < 3; ++c)
    if (!(std_bgr[c] > 0.0f)) return fail(e, YNB_ERR_INVALID, "std must be positive");
  make_prelut(&e->prelut, mean_bgr, std_bgr);
  CUDA_TRY(e, cudaSetDevice(e->cfg.device));
  CUDA_TRY(e, cudaDeviceSynchronize());
  CUDA_TRY(e, cudaMemcpy(e->d_prelut, &e->prelut, sizeof(PreLut), cudaMemcpyHostToDevice));
  return YNB_OK;
}

// Parity hook: the pre-processing alone, device buffers.
YNB_EXPORT int ynb_preprocess_u8(ynb_engine* e, const uint8_t* img_dev, const int32_t* rects_dev, int32_t batch,
                                 float* x_dev, void* stream) {
  if (!e || !img_dev || !x_dev || batch <= 0) return fail(e, YNB_ERR_INVALID, "null argument");
  CUDA_TRY(e, cudaSetDevice(e->cfg.device));
  cudaError_t r = launch_preprocess_u8(img_dev, rects_dev, x_dev, e->d_prelut, batch, e->S, (cudaStream_t)stream);
  if (r != cudaSuccess) return fail(e, YNB_ERR_CUDA, std::string("preprocess_u8: ") + cudaGetErrorString(r));
  return YNB_OK;
}

static_assert(sizeof(ynb_image_desc) == sizeof(ImageDesc), "ynb_image_desc and the kernel's ImageDesc must agree");

YNB_EXPORT int ynb_preprocess_letterbox_u8(ynb_engine* e, const uint8_t* src_dev, const ynb_image_desc* descs_dev,
                                           int32_t batch, float* x_dev, void* stream) {
  if (!e || !src_dev || !descs_dev || !x_dev || batch <= 0) return fail(e, YNB_ERR_INVALID, "null argument");
  CUDA_TRY(e, cudaSetDevice(e->cfg.device));
  cudaError_t r = launch_letterbox_preprocess(src_dev, reinterpret_cast<const ImageDesc*>(descs_dev), x_dev, e->d_prelut,
                                              batch, e->S, (cudaStream_t)stream);
  if (r != cudaSuccess) return fail(e, YNB_ERR_CUDA, std::string("letterbox_preprocess: ") + cudaGetErrorString(r));
  return YNB_OK;
}

YNB_EXPORT int ynb_map_boxes(float* boxes_dev, const int32_t* counts_dev, const double* maps_dev, int32_t batch,
                             int64_t n_per_image, void* stream) {
  if (!boxes_dev || !counts_dev || !maps_dev || batch <= 0 || n_per_image <= 0)
    return fail(nullptr, YNB_ERR_INVALID, "ynb_map_boxes: bad arguments");
  cudaError_t r = launch_map_boxes(boxes_dev, counts_dev, maps_dev, batch, n_per_image, (cudaStream_t)stream);
  if (r != cudaSuccess) return fail(nullptr, YNB_ERR_CUDA, std::string("map_boxes: ") + cudaGetErrorString(r));
  return YNB_OK;
}

// Sorted positions and GT claims are int32 (claims start at 0x7f7f7f7f): the arena stays below that.
constexpr int64_t kVocMaxRows = 0x7f000000;
constexpr int32_t kVocMaxClasses = 4096;

YNB_EXPORT int ynb_voc_append(const float* boxes_dev, const float* scores_dev, const int32_t* cls_dev,
                              const int32_t* counts_dev, int32_t batch, int64_t n_per_image, int32_t image_base,
                              int32_t num_classes, int32_t* rows_dev, int64_t capacity, int64_t* state_dev,
                              void* stream) {
  if (!boxes_dev || !scores_dev || !cls_dev || !counts_dev || !rows_dev || !state_dev || batch <= 0 ||
      n_per_image <= 0 || image_base < 0 || (int64_t)image_base + batch > INT32_MAX || num_classes < 1 ||
      num_classes > kVocMaxClasses || capacity < 0 || capacity > kVocMaxRows)
    return fail(nullptr, YNB_ERR_INVALID, "ynb_voc_append: bad arguments");
  cudaError_t r = ynb::voc::launch_voc_append(boxes_dev, scores_dev, cls_dev, counts_dev, batch, n_per_image,
                                              image_base, num_classes, rows_dev, capacity,
                                              reinterpret_cast<long long*>(state_dev), (cudaStream_t)stream);
  if (r != cudaSuccess) return fail(nullptr, YNB_ERR_CUDA, std::string("voc_append: ") + cudaGetErrorString(r));
  return YNB_OK;
}

YNB_EXPORT int64_t ynb_voc_eval_workspace_bytes(int64_t n_rows, int32_t num_classes, int64_t n_gt) {
  if (n_rows < 0 || n_rows > kVocMaxRows || num_classes < 1 || num_classes > kVocMaxClasses || n_gt < 0) return -1;
  return ynb::voc::eval_workspace(nullptr, n_rows, num_classes, n_gt, nullptr);
}

YNB_EXPORT int ynb_voc_eval(const int32_t* rows_dev, int64_t n_rows, int32_t num_classes, int32_t num_images,
                            const double* gt_boxes_dev, const uint8_t* gt_difficult_dev, const int32_t* gt_start_dev,
                            int64_t n_gt, double ovthresh, int32_t use_07_metric, double* ap_dev, int32_t* npos_dev,
                            int32_t* order_dev, int8_t* flags_dev, void* workspace_dev, int64_t workspace_bytes,
                            void* stream) {
  const int64_t need = ynb_voc_eval_workspace_bytes(n_rows, num_classes, n_gt);
  if (need < 0 || num_images < 0 || (int64_t)num_images * num_classes > INT32_MAX || n_gt > INT32_MAX ||
      (n_rows > 0 && !rows_dev) || (n_gt > 0 && (!gt_boxes_dev || !gt_difficult_dev)) || !gt_start_dev ||
      !ap_dev || !npos_dev || !workspace_dev || workspace_bytes < need)
    return fail(nullptr, YNB_ERR_INVALID, "ynb_voc_eval: bad arguments / workspace too small");
  ynb::voc::EvalWorkspace w;
  ynb::voc::eval_workspace(workspace_dev, n_rows, num_classes, n_gt, &w);
  cudaError_t r = ynb::voc::launch_voc_eval(rows_dev, n_rows, num_classes, num_images, gt_boxes_dev,
                                            gt_difficult_dev, gt_start_dev, n_gt, ovthresh, use_07_metric ? 1 : 0,
                                            ap_dev, npos_dev, order_dev, flags_dev, w, (cudaStream_t)stream);
  if (r != cudaSuccess) return fail(nullptr, YNB_ERR_CUDA, std::string("voc_eval: ") + cudaGetErrorString(r));
  return YNB_OK;
}

YNB_EXPORT int ynb_coco_append(const float* boxes_dev, const float* scores_dev, const int32_t* cls_dev,
                               const int32_t* counts_dev, int32_t batch, int64_t n_per_image, int32_t image_base,
                               int32_t num_classes, int32_t* rows_dev, int64_t capacity, int64_t* state_dev,
                               void* stream) {
  if (!boxes_dev || !scores_dev || !cls_dev || !counts_dev || !rows_dev || !state_dev || batch <= 0 ||
      n_per_image <= 0 || image_base < 0 || (int64_t)image_base + batch > INT32_MAX || num_classes < 1 ||
      num_classes > kVocMaxClasses || capacity < 0 || capacity > kVocMaxRows)
    return fail(nullptr, YNB_ERR_INVALID, "ynb_coco_append: bad arguments");
  cudaError_t r = ynb::coco::launch_coco_append(boxes_dev, scores_dev, cls_dev, counts_dev, batch, n_per_image,
                                                image_base, num_classes, rows_dev, capacity,
                                                reinterpret_cast<long long*>(state_dev), (cudaStream_t)stream);
  if (r != cudaSuccess) return fail(nullptr, YNB_ERR_CUDA, std::string("coco_append: ") + cudaGetErrorString(r));
  return YNB_OK;
}

// Sort keys are uint32 and cell keys image_rank * K + k: the cell count stays below 2^31.
YNB_EXPORT int64_t ynb_coco_eval_workspace_bytes(int64_t n_rows, int32_t num_images, int32_t num_cats,
                                                 int64_t n_gt) {
  if (n_rows < 0 || n_rows > kVocMaxRows || num_images < 0 || num_cats < 1 || num_cats > kVocMaxClasses ||
      (int64_t)num_images * num_cats >= INT32_MAX || n_gt < 0 || n_gt >= INT32_MAX)
    return -1;
  return ynb::coco::eval_workspace(nullptr, n_rows, (int64_t)num_images * num_cats, num_cats, n_gt, nullptr);
}

YNB_EXPORT int ynb_coco_eval(const int32_t* rows_dev, int64_t n_rows, int32_t num_classes, int32_t num_images,
                             const int32_t* image_rank_dev, const int32_t* class_cat_dev, int32_t num_cats,
                             const double* gt_boxes_dev, const double* gt_area_dev, const uint8_t* gt_crowd_dev,
                             const int32_t* gt_start_dev, int64_t n_gt, const double* iou_thrs,
                             const double* rec_thrs, double* precision_dev, double* recall_dev, void* workspace_dev,
                             int64_t workspace_bytes, void* stream) {
  const int64_t need = ynb_coco_eval_workspace_bytes(n_rows, num_images, num_cats, n_gt);
  if (need < 0 || num_classes < 1 || num_classes > kVocMaxClasses || (n_rows > 0 && num_images < 1) ||
      (n_rows > 0 && (!rows_dev || !image_rank_dev)) || !class_cat_dev ||
      (n_gt > 0 && (!gt_boxes_dev || !gt_area_dev || !gt_crowd_dev)) || !gt_start_dev || !iou_thrs || !rec_thrs ||
      !precision_dev || !recall_dev || !workspace_dev || workspace_bytes < need)
    return fail(nullptr, YNB_ERR_INVALID, "ynb_coco_eval: bad arguments / workspace too small");
  ynb::coco::Thresholds thr;
  for (int i = 0; i < ynb::coco::kT; ++i) thr.iou[i] = iou_thrs[i];
  for (int i = 0; i < ynb::coco::kR; ++i) thr.rec[i] = rec_thrs[i];
  ynb::coco::EvalWorkspace w;
  ynb::coco::eval_workspace(workspace_dev, n_rows, (int64_t)num_images * num_cats, num_cats, n_gt, &w);
  cudaError_t r = ynb::coco::launch_coco_eval(rows_dev, n_rows, num_classes, num_images, image_rank_dev,
                                              class_cat_dev, num_cats, gt_boxes_dev, gt_area_dev, gt_crowd_dev,
                                              gt_start_dev, n_gt, thr, precision_dev, recall_dev, w,
                                              (cudaStream_t)stream);
  if (r != cudaSuccess) return fail(nullptr, YNB_ERR_CUDA, std::string("coco_eval: ") + cudaGetErrorString(r));
  return YNB_OK;
}

YNB_EXPORT int ynb_wait_host(ynb_engine* e, int32_t slot_id) {
  if (!e || slot_id < 0 || slot_id > 1) return fail(e, YNB_ERR_INVALID, "bad slot");
  ynb_engine::HostSlot& sl = e->slot[slot_id];
  if (!sl.busy) return fail(e, YNB_ERR_STATE, "nothing submitted on this slot");
  CUDA_TRY(e, cudaSetDevice(e->cfg.device));
  CUDA_TRY(e, cudaEventSynchronize(sl.done));
  sl.busy = false;
  if (*sl.flag_host != 0) {
    int code = *sl.flag_host;
    cudaMemsetAsync(e->d_err, 0, 4, e->s_main);
    return fail(e, YNB_ERR_CUDA, "tensor-core pipeline timed out waiting on mbarrier (code " + std::to_string(code) + ")");
  }
  // counts are on the host now: only the kept rows cross PCIe — three strided copies (rows
  // [0, max count) of every image) on the D2H stream, not 3 x batch small ones behind the next H2D
  const int64_t n = e->N();
  size_t kmax = 0;
  for (int b = 0; b < sl.batch; ++b) kmax = std::max(kmax, (size_t)sl.on[b]);
  if (kmax > 0) {
    CUDA_TRY(e, cudaMemcpy2DAsync(sl.ob, (size_t)n * 16, sl.boxes, (size_t)n * 16, kmax * 16, sl.batch,
                                  cudaMemcpyDeviceToHost, e->s_d2h));
    CUDA_TRY(e, cudaMemcpy2DAsync(sl.os, (size_t)n * 4, sl.scores, (size_t)n * 4, kmax * 4, sl.batch,
                                  cudaMemcpyDeviceToHost, e->s_d2h));
    CUDA_TRY(e, cudaMemcpy2DAsync(sl.oc, (size_t)n * 4, sl.cls, (size_t)n * 4, kmax * 4, sl.batch,
                                  cudaMemcpyDeviceToHost, e->s_d2h));
    CUDA_TRY(e, cudaStreamSynchronize(e->s_d2h));
  }
  return YNB_OK;
}

YNB_EXPORT int ynb_detect_host(ynb_engine* e, const float* x_host, int32_t batch, float* ob, float* os,
                               int32_t* oc, int32_t* on, void* stream) {
  if (!e) return YNB_ERR_INVALID;
  if (e->slot[0].busy) return fail(e, YNB_ERR_STATE, "slot 0 in flight (ynb_submit_host without ynb_wait_host)");
  int rc = ynb_submit_host(e, 0, x_host, batch, ob, os, oc, on, stream);
  return rc ? rc : ynb_wait_host(e, 0);
}

YNB_EXPORT int ynb_tap_shape(const ynb_engine* e, const char* tap, int32_t* c, int32_t* h, int32_t* w) {
  if (!e || !tap || !c || !h || !w) return YNB_ERR_INVALID;
  ynb_engine* me = const_cast<ynb_engine*>(e);
  if (me->taps.empty()) {
    ynb_engine tmp;
    tmp.cfg = e->cfg;
    layout_workspace(&tmp, 1, e->S, nullptr);
    me->taps = tmp.taps;
  }
  auto it = me->taps.find(tap);
  if (it == me->taps.end()) return fail(me, YNB_ERR_INVALID, std::string("unknown tap ") + tap);
  int hh = it->second.H;
  if (me->ws_S != me->S) {   // grid changed since the last forward: rescale
    ynb_engine tmp;
    tmp.cfg = e->cfg;
    layout_workspace(&tmp, 1, e->S, nullptr);
    hh = tmp.taps.at(tap).H;
  }
  *c = it->second.C; *h = hh; *w = hh;
  return YNB_OK;
}

YNB_EXPORT int ynb_read_tap(ynb_engine* e, const char* tap, int32_t batch, float* out_dev, void* stream) {
  if (!e || !tap || !out_dev) return fail(e, YNB_ERR_INVALID, "null argument");
  if (!e->ws || e->ws_S != e->S || batch > e->ws_batch) return fail(e, YNB_ERR_STATE, "run a forward first");
  auto it = e->taps.find(tap);
  if (it == e->taps.end() || !it->second.p) return fail(e, YNB_ERR_INVALID, std::string("unknown tap ") + tap);
  const Tensor& t = it->second;
  CounterScope cs(e);
  int rc = enter(e, (cudaStream_t)stream);
  if (rc) return rc;
  CUDA_TRY(e, launch_nhwc_to_nchw(t.p, t.ld, out_dev, batch, t.C, t.H * t.W, e->s_main, t.es == 2));
  return leave(e, (cudaStream_t)stream);
}

YNB_EXPORT int64_t ynb_launch_count(const ynb_engine* e) { return e ? e->counter.n : 0; }

YNB_EXPORT int ynb_set_profiling(ynb_engine* e, int32_t on) {
  if (!e) return YNB_ERR_INVALID;
  e->profiling = on != 0;
  return YNB_OK;
}

YNB_EXPORT int32_t ynb_profile_count(const ynb_engine* e) { return e ? (int32_t)e->prof.size() : 0; }

YNB_EXPORT int ynb_profile_entry(const ynb_engine* e, int32_t i, const char** name, const char** kind, float* ms,
                                 double* bytes, double* flops) {
  if (!e || i < 0 || i >= (int32_t)e->prof.size() || !name || !kind || !ms || !bytes || !flops) return YNB_ERR_INVALID;
  const ProfEntry& p = e->prof[i];
  *name = p.name.c_str(); *kind = p.kind.c_str(); *ms = p.ms; *bytes = p.bytes; *flops = p.flops;
  return YNB_OK;
}

// ---- unit kernels ------------------------------------------------------------------------------
static thread_local std::string g_unit_error;
#define UNIT_TRY(call)                                                       \
  do {                                                                       \
    cudaError_t _st = (call);                                                \
    if (_st != cudaSuccess) {                                                \
      g_create_error = std::string(#call) + ": " + cudaGetErrorString(_st);  \
      return YNB_ERR_CUDA;                                                   \
    }                                                                        \
  } while (0)

YNB_EXPORT int ynb_dwconv3x3(const float* in, int32_t in_ld, int32_t in_off, float* out, int32_t out_ld,
                             int32_t out_off, int32_t out_step, const float* w, const float* b, int32_t batch,
                             int32_t h_in, int32_t w_in, int32_t channels, int32_t stride, int32_t act, void* stream) {
  if (!in || !out || !w || !b || channels % 4 || in_ld % 4 || in_off % 4 || out_ld % 4 || out_off % 4 ||
      out_step != 1 || (stride != 1 && stride != 2))
    return fail(nullptr, YNB_ERR_INVALID, "ynb_dwconv3x3: channels/ld/off must be multiples of 4, out_step 1");
  CUtensorMap tm;
  if (make_tmap_dw(&tm, in, in_ld, in_off, batch, h_in, w_in, channels, stride)) {
    UNIT_TRY(launch_dwconv3x3_tma(tm, out, out_ld, out_off, w, b, batch, h_in, w_in, channels, stride, act,
                                  (cudaStream_t)stream));
    return YNB_OK;
  }
  UNIT_TRY(launch_dwconv3x3(in, in_ld, in_off, out, out_ld, out_off, w, b, batch, h_in, w_in, channels, stride, act,
                            (cudaStream_t)stream));
  return YNB_OK;
}

// TTA input: bilinear resize (+ flipped copy) of an NCHW float32 batch, device buffers (utils/misc.py:104-121).
YNB_EXPORT int ynb_resize_bilinear(const float* in_dev, int32_t batch, int32_t h_in, int32_t w_in, float* out_dev,
                                   int32_t s_out, int32_t with_flip, void* stream) {
  if (!in_dev || !out_dev || batch <= 0 || h_in <= 0 || w_in <= 0 || s_out <= 0)
    return fail(nullptr, YNB_ERR_INVALID, "ynb_resize_bilinear: bad arguments");
  UNIT_TRY(launch_resize_bilinear(in_dev, out_dev, batch, h_in, w_in, s_out, with_flip, (cudaStream_t)stream));
  return YNB_OK;
}

YNB_EXPORT int ynb_pwconv(const float* in, int32_t in_ld, int32_t in_off, float* out, int32_t out_ld,
                          int32_t out_off, int32_t out_step, const float* w, const float* b, int64_t pixels,
                          int32_t cin, int32_t cout, int32_t act, void* stream) {
  if (!in || !out || !w || !b || cin % 4 || in_ld % 4 || in_off % 4)
    return fail(nullptr, YNB_ERR_INVALID, "ynb_pwconv: cin / in_ld / in_off must be multiples of 4");
  GemmParams g{};
  g.a = in; g.a_ld = in_ld; g.a_off = in_off; g.w = w; g.bias = b; g.out = out; g.out_ld = out_ld;
  g.out_off = out_off; g.out_step = out_step; g.M = pixels; g.N = cout; g.Ktot = cin;
  g.act = act;
  UNIT_TRY(launch_gemm_ffma(g, false, (cudaStream_t)stream));
  return YNB_OK;
}

YNB_EXPORT int ynb_pwconv_tc(const float* in, int32_t in_ld, int32_t in_off, float* out, int32_t out_ld,
                             int32_t out_off, int32_t out_step, const float* w_dev, const float* b_dev,
                             int64_t pixels, int32_t cin, int32_t cout, int32_t act, int32_t mode, void* stream) {
  if (!in || !out || !w_dev || !b_dev || cin % 4 || in_ld % 4 || in_off % 4 || out_ld % 4 ||
      (out_step == 1 && out_off % 4) || cout > 256 || (mode != YNB_GEMM_TC_3XTF32 && mode != YNB_GEMM_TC_TF32))
    return fail(nullptr, YNB_ERR_INVALID, "ynb_pwconv_tc: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  // test hook: pack the weights on the host (synchronous)
  std::vector<float> w((size_t)cout * cin);
  UNIT_TRY(cudaMemcpy(w.data(), w_dev, w.size() * 4, cudaMemcpyDeviceToHost));
  TcWeights t;
  t.N = cout; t.Npad = round_up(cout, 16); t.Kpad = round_up(cin, kTcBK);
  std::vector<float> hi((size_t)t.Npad * t.Kpad, 0.f), lo((size_t)t.Npad * t.Kpad, 0.f);
  for (int n = 0; n < cout; ++n)
    for (int k = 0; k < cin; ++k)
      split_tf32_host(w[(size_t)n * cin + k], &hi[(size_t)n * t.Kpad + k], &lo[(size_t)n * t.Kpad + k]);
  int* d_err = nullptr;
  UNIT_TRY(cudaMalloc(&t.hi, hi.size() * 4));
  UNIT_TRY(cudaMalloc(&t.lo, lo.size() * 4));
  UNIT_TRY(cudaMalloc(&d_err, 4));
  UNIT_TRY(cudaMemset(d_err, 0, 4));
  UNIT_TRY(cudaMemcpy(t.hi, hi.data(), hi.size() * 4, cudaMemcpyHostToDevice));
  UNIT_TRY(cudaMemcpy(t.lo, lo.data(), lo.size() * 4, cudaMemcpyHostToDevice));
  int rc = YNB_OK;
  TcGemmLaunch L;
  L.w = &t;
  TcGemmParams& p = L.p;
  memset(&p, 0, sizeof(p));
  p.mode = mode; p.num_steps = t.Kpad / kTcBK; p.chunks_per_tap = p.num_steps; p.ksub = (cin + 7) / 8;
  p.M = pixels; p.num_tiles = (pixels + kTcBM - 1) / kTcBM; p.N = cout; p.Npad = t.Npad;
  tc_plan_tmem(p);
  p.a_box_bytes = kTcAStageBytes;
  p.out = out; p.out_ld = out_ld; p.out_off = out_off; p.out_step = out_step;
  p.bias = b_dev; p.act = act; p.err_flag = d_err;
  long long* d_trace = nullptr;
  const int trace_cap = 8 * 64 * 32;     // (role, local tile, step) slots, see YNB_TRACE
  const bool want_trace = getenv("YNB_TC_TRACE") != nullptr;
  if (want_trace) {
    UNIT_TRY(cudaMalloc(&d_trace, (1 + 4 * trace_cap) * 8));
    UNIT_TRY(cudaMemset(d_trace, 0, (1 + 4 * trace_cap) * 8));
    p.trace = d_trace; p.trace_cap = trace_cap;
  }
  p.tma_store = (out_step == 1 && out_off % 4 == 0) ? 1 : 0;
  if (getenv("YNB_TC_PASS") != nullptr && cin >= cout && out_ld >= 2 * cout) {
    // timeline hook for the interleave epilogue: pass-through = first `cout` channels of the input rows
    p.pass = in; p.pass_ld = in_ld; p.tma_store = 0; p.out_off = 1; p.out_step = 2;
  }
  if (!make_tmap_2d(&t.tm_hi, t.hi, t.Kpad, t.Npad, t.Kpad, t.Npad) ||
      !make_tmap_2d(&t.tm_lo, t.lo, t.Kpad, t.Npad, t.Kpad, t.Npad) ||
      (p.tma_store && !make_tmap_out(&L.tmOut, out + out_off, (uint64_t)round_up(cout, 4), (uint64_t)pixels,
                                     (uint64_t)out_ld)) ||
      !make_tmap_2d(&L.tmA, in + in_off, cin, pixels, in_ld, kTcBM) || !tc_plan_smem(L)) {
    rc = fail(nullptr, YNB_ERR_CUDA, "ynb_pwconv_tc: tensor map / smem planning failed");
  } else {
    L.grid = (unsigned)std::min<int64_t>(p.num_tiles, kNumSMs);
    cudaError_t r = launch_tc_gemm(L, st);
    if (r == cudaSuccess) r = cudaStreamSynchronize(st);
    int flag = 0;
    if (r == cudaSuccess) r = cudaMemcpy(&flag, d_err, 4, cudaMemcpyDeviceToHost);
    if (r != cudaSuccess) rc = fail(nullptr, YNB_ERR_CUDA, std::string("ynb_pwconv_tc: ") + cudaGetErrorString(r));
    else if (flag) rc = fail(nullptr, YNB_ERR_CUDA, "ynb_pwconv_tc: mbarrier timeout code " + std::to_string(flag));
    if (want_trace && r == cudaSuccess) {
      std::vector<long long> h(1 + 4 * trace_cap);
      cudaMemcpy(h.data(), d_trace, h.size() * 8, cudaMemcpyDeviceToHost);
      int n = 0;
      for (int i = 0; i < trace_cap; ++i) n += h[4 + 4 * i] != 0;
      fprintf(stderr, "YNB_TC_TRACE stages=%d resident=%d nacc=%d acc_stages=%d steps=%d grid=%u events=%d\n",
              p.num_stages, p.w_resident, p.nacc, p.acc_stages, p.num_steps, L.grid, n);
      for (int i = 0; i < trace_cap; ++i)
        if (h[4 + 4 * i] != 0)
          fprintf(stderr, "TRACE %lld %lld %lld %lld\n", h[1 + 4 * i], h[2 + 4 * i], h[3 + 4 * i], h[4 + 4 * i]);
    }
  }
  if (d_trace) cudaFree(d_trace);
  cudaFree(t.hi); cudaFree(t.lo); cudaFree(d_err);
  return rc;
}

YNB_EXPORT int ynb_dwpw_tc(const float* in, int32_t in_ld, const float* dw_w, const float* dw_b, int32_t dw_act,
                           const float* pw_w, const float* pw_b, int32_t act, float* out, int32_t out_ld,
                           const float* pass, int32_t pass_ld, int32_t batch, int32_t h, int32_t w_, int32_t channels,
                           int32_t cout, int32_t mode, void* stream) {
  const bool bfm = mode == YNB_GEMM_TC_BF16;        // in / out / pass are bf16 tensors then (ld in elements, multiples of 8)
  const int al = bfm ? 8 : 4;
  if (!in || !dw_w || !dw_b || !pw_w || !pw_b || !out || channels % al || in_ld % al || out_ld % al || cout > (bfm ? 240 : 128) ||
      cout < 1 || batch < 1 || h < 1 || w_ < 1 ||
      (mode != YNB_GEMM_TC_3XTF32 && mode != YNB_GEMM_TC_TF32 && mode != YNB_GEMM_TC_BF16) ||
      (pass && (out_ld < 2 * cout || pass_ld < cout || pass_ld % 4 || ((uintptr_t)pass & 15u))) || (!pass && out_ld < cout) ||
      ((uintptr_t)out & 15u))
    return fail(nullptr, YNB_ERR_INVALID, "ynb_dwpw_tc: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  std::vector<float> wv((size_t)cout * channels);
  UNIT_TRY(cudaMemcpy(wv.data(), pw_w, wv.size() * 4, cudaMemcpyDeviceToHost));
  TcWeights t;
  t.N = cout; t.Npad = round_up(cout, 16); t.Kpad = round_up(channels, bfm ? 64 : kTcBK);
  std::vector<float> hi((size_t)t.Npad * t.Kpad, 0.f), lo((size_t)t.Npad * t.Kpad, 0.f);
  std::vector<bf16> bwv((size_t)t.Npad * t.Kpad, __float2bfloat16(0.0f));
  for (int n = 0; n < cout; ++n)
    for (int k = 0; k < channels; ++k) {
      split_tf32_host(wv[(size_t)n * channels + k], &hi[(size_t)n * t.Kpad + k], &lo[(size_t)n * t.Kpad + k]);
      bwv[(size_t)n * t.Kpad + k] = __float2bfloat16_rn(wv[(size_t)n * channels + k]);
    }
  int* d_err = nullptr;
  UNIT_TRY(cudaMalloc(&t.hi, hi.size() * 4));
  UNIT_TRY(cudaMalloc(&t.lo, lo.size() * 4));
  UNIT_TRY(cudaMalloc(&d_err, 4));
  UNIT_TRY(cudaMemset(d_err, 0, 4));
  UNIT_TRY(cudaMemcpy(t.hi, hi.data(), hi.size() * 4, cudaMemcpyHostToDevice));
  UNIT_TRY(cudaMemcpy(t.lo, lo.data(), lo.size() * 4, cudaMemcpyHostToDevice));
  if (bfm) UNIT_TRY(cudaMemcpy(t.hi, bwv.data(), bwv.size() * 2, cudaMemcpyHostToDevice));   // one bf16 plane
  int rc = YNB_OK;
  DwPwLaunch L;
  DwPwParams& p = L.p;
  memset(&p, 0, sizeof(p));
  p.dw_w = dw_w; p.dw_b = dw_b; p.dw_act = dw_act;
  p.out = out; p.out_ld = out_ld; p.out_off = 0;
  p.bias = pw_b; p.act = act; p.pass = pass; p.pass_ld = pass ? pass_ld : 0; p.err_flag = d_err;
  long long* d_trace = nullptr;
  const bool want_trace = getenv("YNB_DP_TRACE") != nullptr;
  if (want_trace) {
    UNIT_TRY(cudaMalloc(&d_trace, 6 * 16 * 8 * 8));
    UNIT_TRY(cudaMemset(d_trace, 0, 6 * 16 * 8 * 8));
    p.trace = d_trace;
  }
  if (!make_tmap_2d(&t.tm_hi, t.hi, t.Kpad, t.Npad, t.Kpad, t.Npad, bfm) ||
      !make_tmap_2d(&t.tm_lo, t.lo, t.Kpad, t.Npad, t.Kpad, t.Npad) ||
      !plan_dwpw(L, in, in_ld, batch, h, w_, channels, channels, &t, mode)) {
    rc = fail(nullptr, YNB_ERR_CUDA, "ynb_dwpw_tc: tensor map / smem planning failed");
  } else {
    cudaError_t r = launch_dwpw_tc(L, st);
    if (r == cudaSuccess) r = cudaStreamSynchronize(st);
    int flag = 0;
    if (r == cudaSuccess) r = cudaMemcpy(&flag, d_err, 4, cudaMemcpyDeviceToHost);
    if (r != cudaSuccess) rc = fail(nullptr, YNB_ERR_CUDA, std::string("ynb_dwpw_tc: ") + cudaGetErrorString(r));
    else if (flag) rc = fail(nullptr, YNB_ERR_CUDA, "ynb_dwpw_tc: mbarrier timeout code " + std::to_string(flag));
    if (want_trace && r == cudaSuccess) {
      std::vector<long long> h(6 * 16 * 8);
      cudaMemcpy(h.data(), d_trace, h.size() * 8, cudaMemcpyDeviceToHost);
      long long t0 = 0;
      for (long long v : h) if (v && (!t0 || v < t0)) t0 = v;
      fprintf(stderr, "YNB_DP_TRACE chunks=%d a_stages=%d raw_stages=%d resident=%d lgTW=%d tiles=%lld grid=%u\n", L.p.num_chunks,
              L.p.a_stages, L.p.raw_stages, L.p.w_resident, L.p.lgTW, (long long)L.p.num_tiles, L.grid);
      const char* names[6] = {"raw_issued", "raw_landed", "A_written", "mma_issued", "acc_ready", "epi_done"};
      for (int lt = 0; lt < 16; ++lt)
        for (int role = 0; role < 6; ++role) {
          std::string line;
          for (int kc = 0; kc < 8; ++kc)
            if (h[(role * 16 + lt) * 8 + kc]) line += " " + std::to_string(h[(role * 16 + lt) * 8 + kc] - t0);
          if (!line.empty()) fprintf(stderr, "TRACE tile %2d %-11s%s\n", lt, names[role], line.c_str());
        }
    }
  }
  if (d_trace) cudaFree(d_trace);
  cudaFree(t.hi); cudaFree(t.lo); cudaFree(d_err);
  return rc;
}

YNB_EXPORT int ynb_stem_pool(const float* x, float* out, const float* w, const float* b, int32_t batch,
                             int32_t input_size, void* stream) {
  if (!x || !out || !w || !b || input_size % 32) return fail(nullptr, YNB_ERR_INVALID, "ynb_stem_pool: bad arguments");
  StemWeights wt;   // test hook: fetch the weights into the parameter block (synchronous)
  UNIT_TRY(cudaMemcpy(wt.w, w, sizeof(wt.w), cudaMemcpyDeviceToHost));
  UNIT_TRY(cudaMemcpy(wt.b, b, sizeof(wt.b), cudaMemcpyDeviceToHost));
  CUtensorMap tmx{};
  const int use_tma = make_tmap_stem_input(&tmx, x, input_size, batch) ? 1 : 0;
  UNIT_TRY(launch_stem_pool(x, out, false, wt, tmx, use_tma, batch, input_size, (cudaStream_t)stream));
  return YNB_OK;
}

YNB_EXPORT int ynb_decode_level(const float* raw, int32_t raw_ld, float* boxes, float* scores, int32_t* cls,
                                int32_t batch, int32_t grid, int32_t stride_px, int32_t input_size,
                                const float* anchors_wh, int32_t num_anchors, int32_t num_classes,
                                int64_t boxes_per_image, int64_t level_off, void* stream) {
  if (!raw || !boxes || !scores || !cls || !anchors_wh || num_anchors > 4)
    return fail(nullptr, YNB_ERR_INVALID, "ynb_decode_level: bad arguments");
  DecodeParams d{};
  d.raw = raw; d.ld = raw_ld; d.boxes = boxes; d.scores = scores; d.cls = cls; d.batch = batch; d.G = grid;
  d.A = num_anchors; d.C = num_classes; d.stride = (float)stride_px; d.input_size = (float)input_size;
  for (int a = 0; a < num_anchors; ++a) { d.anchor_w[a] = anchors_wh[2 * a]; d.anchor_h[a] = anchors_wh[2 * a + 1]; }
  d.N = boxes_per_image; d.level_off = level_off;
  UNIT_TRY(launch_decode_level(d, (cudaStream_t)stream));
  return YNB_OK;
}

YNB_EXPORT int64_t ynb_nms_workspace_bytes(int32_t batch, int64_t n) { return nms_workspace_bytes(batch, n); }

YNB_EXPORT int64_t ynb_nms_grid_workspace_bytes(int32_t batch, int32_t input_size) {
  return grid_nms_workspace_bytes(batch, make_grid_geom(input_size).N);
}

YNB_EXPORT int ynb_nms_grid(const float* boxes, const float* scores, const int32_t* cls, int32_t batch,
                            int32_t input_size, int32_t num_classes, float conf, float thr, int32_t diou, float* ob,
                            float* os, int32_t* oc, int32_t* on, uint8_t* keep, void* ws, int64_t ws_bytes,
                            void* stream) {
  if (!boxes || !scores || !cls || !ob || !os || !oc || !on || !ws || input_size <= 0 || input_size % 32 ||
      ws_bytes < ynb_nms_grid_workspace_bytes(batch, input_size))
    return fail(nullptr, YNB_ERR_INVALID, "ynb_nms_grid: bad arguments / workspace too small");
  GridNmsWorkspace w = grid_nms_carve(ws, batch, make_grid_geom(input_size).N);
  UNIT_TRY(launch_nms_grid(boxes, scores, cls, batch, input_size, num_classes, conf, thr, diou, ob, os, oc, on, keep,
                           w, (cudaStream_t)stream));
  return YNB_OK;
}

YNB_EXPORT int ynb_nms(const float* boxes, const float* scores, const int32_t* cls, int32_t batch, int64_t n,
                       int32_t num_classes, float conf, float thr, int32_t diou, float* ob, float* os, int32_t* oc,
                       int32_t* on, uint8_t* keep, void* ws, int64_t ws_bytes, void* stream) {
  if (!boxes || !scores || !cls || !ob || !os || !oc || !on || !ws || ws_bytes < nms_workspace_bytes(batch, n))
    return fail(nullptr, YNB_ERR_INVALID, "ynb_nms: bad arguments / workspace too small");
  NmsWorkspace w = nms_carve(ws, batch, n);
  UNIT_TRY(launch_nms(boxes, scores, cls, batch, n, num_classes, conf, thr, diou, ob, os, oc, on, keep, w,
                      (cudaStream_t)stream));
  return YNB_OK;
}

// ---- training branch at the head boundary (SURVEY §8 row a14 / §8f row 4) ------------------------------

namespace {
bool level_geometry(int input_size, int grid[3], int stride[3]) {
  if (input_size <= 0 || input_size % 32) return false;
  const int st[3] = {8, 16, 32};
  for (int l = 0; l < 3; ++l) { stride[l] = st[l]; grid[l] = input_size / st[l]; }
  return true;
}
}  // namespace

YNB_EXPORT int64_t ynb_train_loss_workspace_bytes(int32_t batch, int32_t input_size) {
  return (int64_t)train_loss_blocks(batch, input_size) * 4 * sizeof(double);
}

YNB_EXPORT int ynb_train_loss(const float* raw_s, const float* raw_m, const float* raw_l, int32_t raw_ld,
                              const float* target, int32_t batch, int32_t input_size, const float* anchors_wh,
                              int32_t num_anchors, int32_t num_classes, float* losses, float* grad_s, float* grad_m,
                              float* grad_l, void* ws, int64_t ws_bytes, void* stream) {
  TrainLossParams p{};
  if (!raw_s || !raw_m || !raw_l || !target || !anchors_wh || !losses || !grad_s || !grad_m || !grad_l || !ws ||
      batch <= 0 || num_anchors <= 0 || num_anchors > kTrainMaxAnchors || num_classes <= 0 ||
      raw_ld < num_anchors * (1 + num_classes + 4) || !level_geometry(input_size, p.grid, p.stride) ||
      ws_bytes < ynb_train_loss_workspace_bytes(batch, input_size))
    return fail(nullptr, YNB_ERR_INVALID, "ynb_train_loss: bad arguments / workspace too small");
  p.raw[0] = raw_s; p.raw[1] = raw_m; p.raw[2] = raw_l;
  p.grad[0] = grad_s; p.grad[1] = grad_m; p.grad[2] = grad_l;
  p.target = target; p.partials = (double*)ws; p.ld = raw_ld; p.B = batch; p.A = num_anchors; p.C = num_classes;
  p.S = input_size;
  int off = 0;
  for (int l = 0; l < 3; ++l) {
    p.cells[l] = p.grid[l] * p.grid[l];
    p.cell_off[l] = off;
    off += p.cells[l];
    for (int a = 0; a < num_anchors; ++a) {
      p.anchors[l][a][0] = anchors_wh[(l * num_anchors + a) * 2];
      p.anchors[l][a][1] = anchors_wh[(l * num_anchors + a) * 2 + 1];
    }
  }
  p.cells_total = off;
  UNIT_TRY(launch_train_loss(p, losses, (cudaStream_t)stream));
  return YNB_OK;
}

YNB_EXPORT int ynb_build_targets(const float* labels, const int32_t* counts, int32_t batch, int32_t max_labels,
                                 int32_t input_size, const float* anchors_wh, int32_t num_anchors, float* target,
                                 void* stream) {
  TargetParams p{};
  if (!labels || !target || !anchors_wh || batch <= 0 || max_labels < 0 || num_anchors <= 0 ||
      num_anchors > kTrainMaxAnchors || !level_geometry(input_size, p.grid, p.stride))
    return fail(nullptr, YNB_ERR_INVALID, "ynb_build_targets: bad arguments");
  p.labels = labels; p.counts = counts; p.target = target; p.B = batch; p.L = max_labels; p.A = num_anchors;
  p.S = input_size;
  long long off = 0;
  for (int l = 0; l < 3; ++l) {
    p.row_off[l] = off;
    off += (long long)p.grid[l] * p.grid[l] * num_anchors;
  }
  p.N = off;
  for (int k = 0; k < 3 * num_anchors; ++k) {
    p.anchors[k][0] = (double)anchors_wh[2 * k];
    p.anchors[k][1] = (double)anchors_wh[2 * k + 1];
  }
  UNIT_TRY(launch_build_targets(p, (cudaStream_t)stream));
  return YNB_OK;
}

YNB_EXPORT int ynb_sgd_step(float* params, const float* grads, float* momentum_buf, int64_t n, float lr,
                            float momentum, float weight_decay, int32_t first_step, float grad_scale, void* stream) {
  if (!params || !grads || !momentum_buf || n <= 0 || ((uintptr_t)params | (uintptr_t)grads | (uintptr_t)momentum_buf) % 16)
    return fail(nullptr, YNB_ERR_INVALID, "ynb_sgd_step: null / unaligned (16 B) buffers");
  UNIT_TRY(launch_sgd_step(params, grads, momentum_buf, n, lr, momentum, weight_decay, first_step, grad_scale,
                           (cudaStream_t)stream));
  return YNB_OK;
}

YNB_EXPORT int32_t ynb_ema_chunk_elems(void) { return kEmaChunk; }

YNB_EXPORT int ynb_ema_update(const uint64_t* ema_ptrs_dev, const uint64_t* model_ptrs_dev, const int64_t* sizes_dev,
                              const int32_t* chunk_tensor_dev, const int32_t* chunk_index_dev, int32_t num_chunks,
                              float d, float one_minus_d, void* stream) {
  if (!ema_ptrs_dev || !model_ptrs_dev || !sizes_dev || !chunk_tensor_dev || !chunk_index_dev || num_chunks < 0)
    return fail(nullptr, YNB_ERR_INVALID, "ynb_ema_update: bad arguments");
  UNIT_TRY(launch_ema_update(reinterpret_cast<const unsigned long long*>(ema_ptrs_dev),
                             reinterpret_cast<const unsigned long long*>(model_ptrs_dev),
                             reinterpret_cast<const long long*>(sizes_dev), chunk_tensor_dev, chunk_index_dev, num_chunks,
                             d, one_minus_d, (cudaStream_t)stream));
  return YNB_OK;
}

YNB_EXPORT int ynb_dwconv3x3_bwd_data(const float* dout, int32_t do_ld, int32_t do_off, float* din, int32_t di_ld,
                                      int32_t di_off, const float* w, int32_t batch, int32_t h_in, int32_t w_in,
                                      int32_t channels, int32_t stride, void* stream) {
  if (!dout || !din || !w || batch <= 0 || h_in <= 0 || w_in <= 0 || channels <= 0 || (stride != 1 && stride != 2))
    return fail(nullptr, YNB_ERR_INVALID, "ynb_dwconv3x3_bwd_data: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  const bool vec = channels % 4 == 0 && do_ld % 4 == 0 && do_off % 4 == 0 && di_ld % 4 == 0 && di_off % 4 == 0 &&
                   ((uintptr_t)dout | (uintptr_t)din | (uintptr_t)w) % 16 == 0;
  CUtensorMap tm;
  if (stride == 1 && vec && make_tmap_dw(&tm, dout, do_ld, do_off, batch, h_in, w_in, channels, 1)) {
    // stride 1: the forward convolution of d_out with the taps reversed, on the TMA halo-tile kernel
    UNIT_TRY(launch_dwconv3x3_tma(tm, din, di_ld, di_off, w, nullptr, batch, h_in, w_in, channels, 1, YNB_ACT_NONE, st,
                                  /*reversed_taps=*/true));
    return YNB_OK;
  }
  if (stride == 2 && vec && 9 * channels * 4 <= 48 * 1024) {
    const long long items = (long long)batch * ((h_in + 1) / 2) * ((w_in + 1) / 2) * (channels / 4);
    const int nb = (int)std::min<long long>((items + 255) / 256, (long long)kNumSMs * 8);
    dwconv3x3_s2_bwd_data_kernel<<<nb, 256, 9 * channels * sizeof(float), st>>>(dout, do_ld, do_off, din, di_ld, di_off, w,
                                                                               batch, h_in, w_in, channels);
    YNB_COUNT_LAUNCH();
    UNIT_TRY(cudaGetLastError());
    return YNB_OK;
  }
  const long long total = (long long)batch * h_in * w_in * ((channels + 3) / 4);
  const int blocks = (int)std::min<long long>((total + 255) / 256, (long long)kNumSMs * 16);
  if (vec)
    dwconv3x3_bwd_data_kernel<true><<<blocks, 256, 0, st>>>(dout, do_ld, do_off, din, di_ld, di_off, w, batch, h_in, w_in,
                                                            channels, stride);
  else
    dwconv3x3_bwd_data_kernel<false><<<blocks, 256, 0, st>>>(dout, do_ld, do_off, din, di_ld, di_off, w, batch, h_in, w_in,
                                                             channels, stride);
  YNB_COUNT_LAUNCH();
  UNIT_TRY(cudaGetLastError());
  return YNB_OK;
}

YNB_EXPORT int64_t ynb_dwconv3x3_bwd_weight_workspace_bytes(int32_t batch, int32_t h_in, int32_t w_in, int32_t channels,
                                                            int32_t stride) {
  const int h_out = (h_in - 1) / stride + 1, w_out = (w_in - 1) / stride + 1;
  return (int64_t)dw_bwd_chunks(batch, h_out, w_out) * 10 * channels * sizeof(float);
}

YNB_EXPORT int ynb_dwconv3x3_bwd_weight(const float* dout, int32_t do_ld, int32_t do_off, const float* in, int32_t in_ld,
                                        int32_t in_off, float* dwdb, int32_t batch, int32_t h_in, int32_t w_in,
                                        int32_t channels, int32_t stride, void* ws, int64_t ws_bytes, void* stream) {
  if (!dout || !in || !dwdb || !ws || batch <= 0 || h_in <= 0 || w_in <= 0 || channels <= 0 ||
      (stride != 1 && stride != 2) ||
      ws_bytes < ynb_dwconv3x3_bwd_weight_workspace_bytes(batch, h_in, w_in, channels, stride))
    return fail(nullptr, YNB_ERR_INVALID, "ynb_dwconv3x3_bwd_weight: bad arguments / workspace too small");
  const int h_out = (h_in - 1) / stride + 1, w_out = (w_in - 1) / stride + 1;
  const int chunks = dw_bwd_chunks(batch, h_out, w_out);
  const bool vec = channels % 4 == 0 && do_ld % 4 == 0 && do_off % 4 == 0 && in_ld % 4 == 0 && in_off % 4 == 0 &&
                   ((uintptr_t)dout | (uintptr_t)in) % 16 == 0;
  dim3 grid(chunks, (channels + kDwBwdCg * 4 - 1) / (kDwBwdCg * 4)), block(kDwBwdCg, kDwBwdSlices);
  cudaStream_t st = (cudaStream_t)stream;
  float* part = (float*)ws;
#define YNB_DWBW(S, V) \
  dwconv3x3_bwd_weight_kernel<S, V><<<grid, block, 0, st>>>(dout, do_ld, do_off, in, in_ld, in_off, part, batch, h_in, w_in, channels)
  if (stride == 1) { if (vec) YNB_DWBW(1, true); else YNB_DWBW(1, false); }
  else             { if (vec) YNB_DWBW(2, true); else YNB_DWBW(2, false); }
#undef YNB_DWBW
  YNB_COUNT_LAUNCH();
  launch_reduce_partials(part, chunks, 10LL * channels, dwdb, st);
  UNIT_TRY(cudaGetLastError());
  return YNB_OK;
}

YNB_EXPORT int64_t ynb_pwconv_bwd_weight_workspace_bytes(int64_t pixels, int32_t cin, int32_t cout) {
  int64_t floats = (int64_t)pw_bwd_chunks(pixels, cin, cout) * ((int64_t)cout * cin + cout);
  if (wgrad_tc_kpad(cin)) floats = std::max<int64_t>(floats, wgrad_tc_partial_floats(pixels, cin, cout));
  return floats * sizeof(float) + 16;     // + the device error word
}

YNB_EXPORT int ynb_pwconv_bwd_weight(const float* dout, int32_t do_ld, int32_t do_off, const float* in, int32_t in_ld,
                                     int32_t in_off, float* dw, float* db, int64_t pixels, int32_t cin, int32_t cout,
                                     void* ws, int64_t ws_bytes, void* stream) {
  if (!dout || !in || !dw || !db || !ws || pixels <= 0 || cin <= 0 || cout <= 0 ||
      ws_bytes < ynb_pwconv_bwd_weight_workspace_bytes(pixels, cin, cout))
    return fail(nullptr, YNB_ERR_INVALID, "ynb_pwconv_bwd_weight: bad arguments / workspace too small");
  const bool aligned = cin % 4 == 0 && cout % 4 == 0 && do_ld % 4 == 0 && do_off % 4 == 0 && in_ld % 4 == 0 &&
                       in_off % 4 == 0 && ((uintptr_t)dout | (uintptr_t)in) % 16 == 0;
  if (wgrad_tc_kpad(cin) != 0 && aligned) {
    // tcgen05 path (3xTF32 = fp32 parity): pixels are the contraction dimension
    cudaStream_t st = (cudaStream_t)stream;
    const int chunks = wgrad_tc_chunks(pixels, cout);
    int* err = (int*)((char*)ws + ynb_pwconv_bwd_weight_workspace_bytes(pixels, cin, cout) - 16);
    UNIT_TRY(cudaMemsetAsync(err, 0, 4, st));
    WgradParams p{};
    p.dout = dout; p.do_ld = do_ld; p.do_off = do_off; p.in = in; p.in_ld = in_ld; p.in_off = in_off;
    p.partial = (float*)ws; p.M = pixels; p.K = cin; p.N = cout; p.err = err;
    UNIT_TRY(launch_pw_wgrad_tc(p, chunks, st));
    {
      const int ntiles = (cout + 127) / 128, kpad = wgrad_tc_kpad(cin);
      const long long elems = (long long)ntiles * 128 * kpad;
      launch_wgrad_reduce((const float*)ws, chunks, ntiles, kpad, cout, cin, dw, db, st);
      YNB_COUNT_LAUNCH();
    }
    UNIT_TRY(cudaGetLastError());
    if (getenv("YNB_SYNC_CHECK")) {          // tests: surface a bounded-wait timeout instead of wrong numbers
      int flag = 0;
      UNIT_TRY(cudaStreamSynchronize(st));
      UNIT_TRY(cudaMemcpy(&flag, err, 4, cudaMemcpyDeviceToHost));
      if (flag) return fail(nullptr, YNB_ERR_CUDA, "ynb_pwconv_bwd_weight: mbarrier timeout code " + std::to_string(flag));
    }
    return YNB_OK;
  }
  const int chunks = pw_bwd_chunks(pixels, cin, cout);
  long long m_per_chunk = (pixels + chunks - 1) / chunks;
  m_per_chunk = (m_per_chunk + kPwBwdSlab - 1) / kPwBwdSlab * kPwBwdSlab;
  float* pw = (float*)ws;
  float* pb = pw + (long long)chunks * cout * cin;
  cudaStream_t st = (cudaStream_t)stream;
  // a chunk past the end of M (rounding of m_per_chunk) writes zeros: no memset needed
  dim3 grid(chunks, (cout + kPwBwdTile - 1) / kPwBwdTile, (cin + kPwBwdTile - 1) / kPwBwdTile);
  if (aligned) {
    // per device, cheap: set on every call (one process may drive several devices)
    UNIT_TRY(cudaFuncSetAttribute(pwconv_bwd_weight_async_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)kPwBwdAsyncSmem));
    pwconv_bwd_weight_async_kernel<<<grid, 256, kPwBwdAsyncSmem, st>>>(dout, do_ld, do_off, in, in_ld, in_off, pw, pb,
                                                                       pixels, cin, cout, m_per_chunk);
  } else {
    pwconv_bwd_weight_kernel<<<grid, 256, 0, st>>>(dout, do_ld, do_off, in, in_ld, in_off, pw, pb, pixels, cin, cout,
                                                   m_per_chunk);
  }
  YNB_COUNT_LAUNCH();
  launch_reduce_partials(pw, chunks, (long long)cout * cin, dw, st);
  launch_reduce_partials(pb, chunks, cout, db, st);
  UNIT_TRY(cudaGetLastError());
  return YNB_OK;
}

YNB_EXPORT int ynb_act_bwd(const float* dout, int32_t do_ld, int32_t do_off, const float* out, int32_t o_ld,
                           int32_t o_off, float* dpre, int32_t dp_ld, int32_t dp_off, int64_t pixels, int32_t channels,
                           int32_t act, void* stream) {
  if (!dout || !out || !dpre || pixels <= 0 || channels <= 0 || (act != YNB_ACT_RELU && act != YNB_ACT_LEAKY))
    return fail(nullptr, YNB_ERR_INVALID, "ynb_act_bwd: bad arguments");
  const long long total = (long long)pixels * channels;
  const int blocks = (int)std::min<long long>((total + 255) / 256, (long long)kNumSMs * 16);
  act_bwd_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(dout, do_ld, do_off, out, o_ld, o_off, dpre, dp_ld, dp_off,
                                                           pixels, channels, act == YNB_ACT_RELU ? 0.0f : 0.1f);
  YNB_COUNT_LAUNCH();
  UNIT_TRY(cudaGetLastError());
  return YNB_OK;
}

// YOLONano.forward(x, target) with trainable = True and the BatchNorm layers in eval mode (running
// statistics: the network part is the inference network): backbone + neck + heads on the tensor-core
// path, then the loss / gradient kernel directly on the engine's NHWC head maps (no permute, no copy).
YNB_EXPORT int ynb_forward_train_loss(ynb_engine* e, const float* x_dev, int32_t batch, const float* target,
                                      float* losses, float* grad_s, float* grad_m, float* grad_l, void* ws,
                                      int64_t ws_bytes, void* stream) {
  if (!e || !x_dev || !target || !losses || !grad_s || !grad_m || !grad_l || !ws)
    return fail(e, YNB_ERR_INVALID, "null argument");
  if (ws_bytes < ynb_train_loss_workspace_bytes(batch, e->S))
    return fail(e, YNB_ERR_INVALID, "ynb_forward_train_loss: workspace too small");
  cudaStream_t user = (cudaStream_t)stream;
  CounterScope cs(e);
  Plan* plan = nullptr;
  int rc = prepare(e, batch, &plan);
  if (rc || (rc = enter(e, user)) || (rc = run_network(e, x_dev, plan))) return rc;
  TrainLossParams p{};
  level_geometry(e->S, p.grid, p.stride);   // the CURRENT grid (ynb_set_grid), not the creation-time one
  float* grads[3] = {grad_s, grad_m, grad_l};
  int off = 0;
  for (int l = 0; l < 3; ++l) {
    p.raw[l] = e->raw[l].p; p.grad[l] = grads[l];
    p.cells[l] = p.grid[l] * p.grid[l];
    p.cell_off[l] = off;
    off += p.cells[l];
    for (int a = 0; a < e->cfg.num_anchors; ++a) {
      p.anchors[l][a][0] = e->cfg.anchors[(l * e->cfg.num_anchors + a) * 2];
      p.anchors[l][a][1] = e->cfg.anchors[(l * e->cfg.num_anchors + a) * 2 + 1];
    }
  }
  p.cells_total = off;
  p.target = target; p.partials = (double*)ws; p.ld = e->raw[0].ld; p.B = batch; p.A = e->cfg.num_anchors;
  p.C = e->cfg.num_classes; p.S = e->S;
  if (p.ld != ynb_raw_ld(e)) return fail(e, YNB_ERR_STATE, "ynb_forward_train_loss: head map stride changed");
  CUDA_TRY(e, launch_train_loss(p, losses, e->s_main));
  if ((rc = leave(e, user))) return rc;
  return e->cfg.gemm_mode == YNB_GEMM_FP32_FFMA ? YNB_OK : check_device_error(e);
}

YNB_EXPORT int32_t ynb_raw_ld(const ynb_engine* e) {
  return e ? round_up(e->cfg.num_anchors * (1 + e->cfg.num_classes + 4), 4) : 0;   // = plan_workspace's raw[l].ld
}

// Weight gradient of a dense 3x3 conv (pad 1, stride 1: the four `smooth` convs, models/yolo_nano.py:44-47):
// nine tap-shifted pointwise weight gradients on the tcgen05 kernel, dW[t][n][k] = sum_m dY[m][n] * X[m + tap_t][k]
// with X = 0 outside the image.
YNB_EXPORT int ynb_conv3x3_bwd_weight(const float* dout, int32_t do_ld, int32_t do_off, const float* in, int32_t in_ld,
                                      int32_t in_off, float* dw9, float* db, int32_t batch, int32_t h, int32_t w_,
                                      int32_t cin, int32_t cout, void* ws, int64_t ws_bytes, void* stream) {
  const int64_t pixels = (int64_t)batch * h * w_;
  const bool aligned = cin % 4 == 0 && cout % 4 == 0 && do_ld % 4 == 0 && do_off % 4 == 0 && in_ld % 4 == 0 &&
                       in_off % 4 == 0 && ((uintptr_t)dout | (uintptr_t)in) % 16 == 0;
  if (!dout || !in || !dw9 || !db || !ws || batch <= 0 || h <= 0 || w_ <= 0 || cin <= 0 || cout <= 0 ||
      pixels >= (1LL << 31) || ws_bytes < ynb_pwconv_bwd_weight_workspace_bytes(pixels, cin, cout))
    return fail(nullptr, YNB_ERR_INVALID, "ynb_conv3x3_bwd_weight: bad arguments / workspace too small");
  if (!aligned || !wgrad_tc_kpad(cin))
    return fail(nullptr, YNB_ERR_UNSUPPORTED, "ynb_conv3x3_bwd_weight: needs 16-byte aligned views and cin <= 255");
  cudaStream_t st = (cudaStream_t)stream;
  const int chunks = wgrad_tc_chunks(pixels, cout);
  int* err = (int*)((char*)ws + ynb_pwconv_bwd_weight_workspace_bytes(pixels, cin, cout) - 16);
  UNIT_TRY(cudaMemsetAsync(err, 0, 4, st));
  const int ntiles = (cout + 127) / 128, kpad = wgrad_tc_kpad(cin);
  const long long elems = (long long)ntiles * 128 * kpad;
  for (int t = 0; t < 9; ++t) {
    WgradParams p{};
    p.dout = dout; p.do_ld = do_ld; p.do_off = do_off; p.in = in; p.in_ld = in_ld; p.in_off = in_off;
    p.partial = (float*)ws; p.M = pixels; p.K = cin; p.N = cout; p.err = err;
    p.H = h; p.W = w_; p.dy = t / 3 - 1; p.dx = t % 3 - 1;
    UNIT_TRY(launch_pw_wgrad_tc(p, chunks, st));
    launch_wgrad_reduce((const float*)ws, chunks, ntiles, kpad, cout, cin, dw9 + (long long)t * cout * cin, db, st);
    YNB_COUNT_LAUNCH();
  }
  UNIT_TRY(cudaGetLastError());
  if (getenv("YNB_SYNC_CHECK")) {
    int flag = 0;
    UNIT_TRY(cudaStreamSynchronize(st));
    UNIT_TRY(cudaMemcpy(&flag, err, 4, cudaMemcpyDeviceToHost));
    if (flag) return fail(nullptr, YNB_ERR_CUDA, "ynb_conv3x3_bwd_weight: mbarrier timeout code " + std::to_string(flag));
  }
  return YNB_OK;
}

// ---- round 2: entries of the chained training step (yolo_nano_b200/train_step.py) ------------------------------
YNB_EXPORT int ynb_stem_conv_fwd(const float* x, const float* w2724, float* out, int32_t batch, int32_t input_size,
                                 void* stream) {
  if (!x || !w2724 || !out || batch <= 0 || input_size <= 0 || input_size % 2)
    return fail(nullptr, YNB_ERR_INVALID, "ynb_stem_conv_fwd: bad arguments");
  const long long items = (long long)batch * (input_size / 2) * (input_size / 2) * 6;
  stem_conv_fwd_kernel<<<grid_for(items), 256, 0, (cudaStream_t)stream>>>(x, w2724, out, batch, input_size);
  YNB_COUNT_LAUNCH();
  UNIT_TRY(cudaGetLastError());
  return YNB_OK;
}

YNB_EXPORT int64_t ynb_stem_conv_bwd_weight_workspace_bytes(int32_t batch, int32_t input_size) {
  return (int64_t)stem_wg_chunks(batch, input_size) * kStemWgOut * sizeof(float);
}

YNB_EXPORT int ynb_stem_conv_bwd_weight(const float* dout, const float* x, float* dw2724, int32_t batch, int32_t input_size,
                                        void* ws, int64_t ws_bytes, void* stream) {
  if (!dout || !x || !dw2724 || !ws || batch <= 0 || input_size <= 0 || input_size % 2 ||
      ws_bytes < ynb_stem_conv_bwd_weight_workspace_bytes(batch, input_size))
    return fail(nullptr, YNB_ERR_INVALID, "ynb_stem_conv_bwd_weight: bad arguments / workspace too small");
  if (((uintptr_t)dout | (uintptr_t)ws) & 15u)
    return fail(nullptr, YNB_ERR_INVALID, "ynb_stem_conv_bwd_weight: dout / workspace must be 16-byte aligned");
  const int grid = stem_wg_grid(batch, input_size), nseg = stem_wg_nseg(input_size);
  const long long items = (long long)batch * (input_size / 2) * nseg;
  if (items > INT32_MAX) return fail(nullptr, YNB_ERR_INVALID, "ynb_stem_conv_bwd_weight: batch too large");
  cudaStream_t st = (cudaStream_t)stream;
  stem_conv_bwd_weight_kernel<<<grid, kStemWgThreads, 0, st>>>(dout, x, (float*)ws, batch, input_size, (int)items, nseg);
  YNB_COUNT_LAUNCH();
  launch_reduce_partials((const float*)ws, 2 * grid, kStemWgOut, dw2724, st);
  UNIT_TRY(cudaGetLastError());
  return YNB_OK;
}

YNB_EXPORT int ynb_maxpool3x3s2_fwd(const float* in, float* out, int32_t batch, int32_t h, int32_t w_, int32_t channels,
                                    void* stream) {
  if (!in || !out || batch <= 0 || h <= 0 || w_ <= 0 || channels <= 0 || channels % 4)
    return fail(nullptr, YNB_ERR_INVALID, "ynb_maxpool3x3s2_fwd: bad arguments");
  const long long items = (long long)batch * ((h - 1) / 2 + 1) * ((w_ - 1) / 2 + 1) * (channels / 4);
  maxpool3x3s2_fwd_kernel<<<grid_for(items), 256, 0, (cudaStream_t)stream>>>(in, out, batch, h, w_, channels);
  YNB_COUNT_LAUNCH();
  UNIT_TRY(cudaGetLastError());
  return YNB_OK;
}

YNB_EXPORT int ynb_maxpool3x3s2_bwd(const float* dout, const float* in, float* din, int32_t batch, int32_t h, int32_t w_,
                                    int32_t channels, void* stream) {
  if (!dout || !in || !din || batch <= 0 || h <= 0 || w_ <= 0 || channels <= 0)
    return fail(nullptr, YNB_ERR_INVALID, "ynb_maxpool3x3s2_bwd: bad arguments");
  const long long items = (long long)batch * h * w_ * channels;
  maxpool3x3s2_bwd_kernel<<<grid_for(items), 256, 0, (cudaStream_t)stream>>>(dout, in, din, batch, h, w_, channels);
  YNB_COUNT_LAUNCH();
  UNIT_TRY(cudaGetLastError());
  return YNB_OK;
}

YNB_EXPORT int ynb_shuffle_unit_move(float* x, float* a, float* b, int64_t rows, int32_t half, int32_t half_padded,
                                     int32_t op, void* stream) {
  if (!x || !a || !b || rows <= 0 || half <= 0 || half_padded < half || op < 0 || op > 3 || (((uintptr_t)x) & 7u))
    return fail(nullptr, YNB_ERR_INVALID, "ynb_shuffle_unit_move: bad arguments");
  shuffle_unit_move_kernel<<<grid_for(rows * half_padded), 256, 0, (cudaStream_t)stream>>>(x, a, b, rows, half, half_padded, op);
  YNB_COUNT_LAUNCH();
  UNIT_TRY(cudaGetLastError());
  return YNB_OK;
}

YNB_EXPORT int ynb_maxpool3x3s2_fwd_idx(const float* in, float* out, uint8_t* idx, int32_t batch, int32_t h, int32_t w_,
                                        int32_t channels, void* stream) {
  if (!in || !out || !idx || batch <= 0 || h <= 0 || w_ <= 0 || channels <= 0 || channels % 4 ||
      (((uintptr_t)in | (uintptr_t)out) & 15u) || ((uintptr_t)idx & 3u))
    return fail(nullptr, YNB_ERR_INVALID, "ynb_maxpool3x3s2_fwd_idx: bad arguments");
  const long long items = (long long)batch * ((h - 1) / 2 + 1) * ((w_ - 1) / 2 + 1) * (channels / 4);
  maxpool3x3s2_fwd_idx_kernel<<<grid_for(items), 256, 0, (cudaStream_t)stream>>>(in, out, idx, batch, h, w_, channels);
  YNB_COUNT_LAUNCH();
  UNIT_TRY(cudaGetLastError());
  return YNB_OK;
}

YNB_EXPORT int ynb_maxpool3x3s2_bwd_idx(const float* dout, const uint8_t* idx, float* din, int32_t batch, int32_t h,
                                        int32_t w_, int32_t channels, void* stream) {
  if (!dout || !idx || !din || batch <= 0 || h <= 0 || w_ <= 0 || channels <= 0 || channels % 4 ||
      (((uintptr_t)dout | (uintptr_t)din) & 15u) || ((uintptr_t)idx & 3u))
    return fail(nullptr, YNB_ERR_INVALID, "ynb_maxpool3x3s2_bwd_idx: bad arguments");
  const long long items = (long long)batch * h * w_ * (channels / 4);
  maxpool3x3s2_bwd_idx_kernel<<<grid_for(items), 256, 0, (cudaStream_t)stream>>>(dout, idx, din, batch, h, w_, channels);
  YNB_COUNT_LAUNCH();
  UNIT_TRY(cudaGetLastError());
  return YNB_OK;
}

YNB_EXPORT int ynb_resample_add(const float* a, const float* a2, float* out, int32_t batch, int32_t h, int32_t w_,
                                int32_t channels, int32_t mode, void* stream) {
  if (!a || !a2 || !out || batch <= 0 || h <= 0 || w_ <= 0 || channels <= 0 || channels % 4 || (mode != 1 && mode != 2) ||
      (mode == 1 && ((h | w_) & 1)))
    return fail(nullptr, YNB_ERR_INVALID, "ynb_resample_add: bad arguments");
  UNIT_TRY(launch_resample_add(a, a2, out, nullptr, batch, h, w_, channels, mode, (cudaStream_t)stream));
  return YNB_OK;
}

YNB_EXPORT int ynb_resample_bwd(const float* dout, float* da2, int32_t batch, int32_t h, int32_t w_, int32_t channels,
                                int32_t mode, void* stream) {
  if (!dout || !da2 || batch <= 0 || h <= 0 || w_ <= 0 || channels <= 0 || channels % 4 || (mode != 1 && mode != 2) ||
      (mode == 1 && ((h | w_) & 1)))
    return fail(nullptr, YNB_ERR_INVALID, "ynb_resample_bwd: bad arguments");
  const int h2 = mode == 1 ? h / 2 : h * 2, w2 = mode == 1 ? w_ / 2 : w_ * 2;
  const long long items = (long long)batch * h2 * w2 * (channels / 4);
  resample_bwd_kernel<<<grid_for(items), 256, 0, (cudaStream_t)stream>>>(dout, da2, batch, h, w_, channels, mode);
  YNB_COUNT_LAUNCH();
  UNIT_TRY(cudaGetLastError());
  return YNB_OK;
}

YNB_EXPORT int ynb_add(const float* a, const float* b, float* out, int64_t n, void* stream) {
  if (!a || !b || !out || n <= 0 || n % 4 || (((uintptr_t)a | (uintptr_t)b | (uintptr_t)out) & 15u))
    return fail(nullptr, YNB_ERR_INVALID, "ynb_add: n must be a multiple of 4, buffers 16-byte aligned");
  add_kernel<<<grid_for(n / 4), 256, 0, (cudaStream_t)stream>>>(a, b, out, n / 4);
  YNB_COUNT_LAUNCH();
  UNIT_TRY(cudaGetLastError());
  return YNB_OK;
}

// Dense 3x3 conv, pad 1, stride 1, + bias + activation on the tcgen05 implicit-GEMM path (3xTF32 | TF32), standalone:
// forward of the `smooth` convs (models/yolo_nano.py:44-47) and, with w'[k][8 - t][n] = w[n][t][k], their input
// gradient.  w_dev [cout][9][cin] tap-major (cin % 32 == 0, cout <= 256).  Synchronous test / training hook (packs the
// weights on the host, like ynb_pwconv_tc).
YNB_EXPORT int ynb_conv3x3_tc(const float* in, int32_t in_ld, float* out, int32_t out_ld, const float* w_dev,
                              const float* b_dev, int32_t batch, int32_t h, int32_t w_, int32_t cin, int32_t cout,
                              int32_t act, int32_t mode, void* stream) {
  if (!in || !out || !w_dev || !b_dev || batch <= 0 || h <= 0 || w_ <= 0 || cin <= 0 || cin % kTcBK || in_ld % 4 ||
      out_ld % 4 || cout < 1 || cout > 256 || (mode != YNB_GEMM_TC_3XTF32 && mode != YNB_GEMM_TC_TF32) ||
      (((uintptr_t)in | (uintptr_t)out) & 15u))
    return fail(nullptr, YNB_ERR_INVALID, "ynb_conv3x3_tc: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  const int ktot = 9 * cin;
  std::vector<float> wv((size_t)cout * ktot);
  UNIT_TRY(cudaMemcpy(wv.data(), w_dev, wv.size() * 4, cudaMemcpyDeviceToHost));
  TcWeights t;
  t.N = cout; t.Npad = round_up(cout, 16); t.Kpad = ktot;
  std::vector<float> hi((size_t)t.Npad * t.Kpad, 0.f), lo((size_t)t.Npad * t.Kpad, 0.f);
  for (int n = 0; n < cout; ++n)
    for (int k = 0; k < ktot; ++k)
      split_tf32_host(wv[(size_t)n * ktot + k], &hi[(size_t)n * t.Kpad + k], &lo[(size_t)n * t.Kpad + k]);
  int* d_err = nullptr;
  UNIT_TRY(cudaMalloc(&t.hi, hi.size() * 4));
  UNIT_TRY(cudaMalloc(&t.lo, lo.size() * 4));
  UNIT_TRY(cudaMalloc(&d_err, 4));
  UNIT_TRY(cudaMemset(d_err, 0, 4));
  UNIT_TRY(cudaMemcpy(t.hi, hi.data(), hi.size() * 4, cudaMemcpyHostToDevice));
  UNIT_TRY(cudaMemcpy(t.lo, lo.data(), lo.size() * 4, cudaMemcpyHostToDevice));
  int rc = YNB_OK;
  TcGemmLaunch L;
  L.w = &t;
  TcGemmParams& p = L.p;
  memset(&p, 0, sizeof(p));
  p.mode = mode; p.is3x3 = 1;
  p.chunks_per_tap = cin / kTcBK;
  p.num_steps = 9 * p.chunks_per_tap;
  p.H = h; p.W = w_;
  tc_pick_tile(p.H, p.W, &p.TH, &p.TW);
  p.tiles_x = (p.W + p.TW - 1) / p.TW;
  p.tiles_y = (p.H + p.TH - 1) / p.TH;
  p.num_tiles = (int64_t)batch * p.tiles_x * p.tiles_y;
  p.M = (int64_t)batch * h * w_;
  p.N = cout; p.Npad = t.Npad;
  tc_plan_tmem(p);
  p.a_box_bytes = (uint32_t)(p.TH * p.TW * 128);
  p.out = out; p.out_ld = out_ld; p.out_off = 0; p.out_step = 1;
  p.bias = b_dev; p.act = act; p.err_flag = d_err;
  if (!make_tmap_2d(&t.tm_hi, t.hi, t.Kpad, t.Npad, t.Kpad, t.Npad) ||
      !make_tmap_2d(&t.tm_lo, t.lo, t.Kpad, t.Npad, t.Kpad, t.Npad) ||
      !make_tmap_nhwc(&L.tmA, in, cin, w_, h, batch, in_ld, p.TW, p.TH) || !tc_plan_smem(L)) {
    rc = fail(nullptr, YNB_ERR_CUDA, "ynb_conv3x3_tc: tensor map / smem planning failed");
  } else {
    L.grid = (unsigned)std::min<int64_t>(p.num_tiles, kNumSMs);
    cudaError_t r = launch_tc_gemm(L, st);
    if (r == cudaSuccess) r = cudaStreamSynchronize(st);
    int flag = 0;
    if (r == cudaSuccess) r = cudaMemcpy(&flag, d_err, 4, cudaMemcpyDeviceToHost);
    if (r != cudaSuccess) rc = fail(nullptr, YNB_ERR_CUDA, std::string("ynb_conv3x3_tc: ") + cudaGetErrorString(r));
    else if (flag) rc = fail(nullptr, YNB_ERR_CUDA, "ynb_conv3x3_tc: mbarrier timeout code " + std::to_string(flag));
  }
  cudaFree(t.hi); cudaFree(t.lo); cudaFree(d_err);
  return rc;
}

// ---- training-grade tensor-core convs: asynchronous, no allocation, weights packed on the device -------------
// The `ynb_pwconv_tc` / `ynb_conv3x3_tc` hooks above pack the weights on the host and synchronise (they exist for
// the kernel unit tests).  A training step changes every weight every iteration, so here the hi / lo TF32 planes are
// produced by a kernel into a caller-provided workspace, right before the GEMM on the same stream; nothing blocks.
namespace {
// w element (n, k) = trans ? w[k * w_ld + n] : w[n * w_ld + k]; zero outside rows x cols.
__global__ void pack_tc_weights_kernel(const float* __restrict__ w, int w_ld, int rows, int cols, int trans,
                                       float* __restrict__ hi, float* __restrict__ lo, int Npad, int Kpad, int* err_flag) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0 && err_flag) *err_flag = 0;
  if (i >= Npad * Kpad) return;
  const int n = i / Kpad, k = i - n * Kpad;
  float v = 0.f;
  if (n < rows && k < cols) v = trans ? w[(size_t)k * w_ld + n] : w[(size_t)n * w_ld + k];
  const uint32_t h = rn_tf32_bits(__float_as_uint(v));
  hi[i] = __uint_as_float(h);
  lo[i] = __uint_as_float(rn_tf32_bits(__float_as_uint(v - __uint_as_float(h))));
}

struct AsyncWs { float* hi; float* lo; int* flag; };
int64_t tc_async_bytes(int Npad, int Kpad) { return (int64_t)2 * Npad * Kpad * 4 + 256; }
bool carve_async(void* ws, int64_t bytes, int Npad, int Kpad, AsyncWs* o) {
  if (!ws || ((uintptr_t)ws & 255u) || bytes < tc_async_bytes(Npad, Kpad)) return false;
  o->hi = (float*)ws;
  o->lo = o->hi + (size_t)Npad * Kpad;
  o->flag = (int*)(o->lo + (size_t)Npad * Kpad);
  return true;
}
}  // namespace

YNB_EXPORT int64_t ynb_tc_async_workspace_bytes(int32_t cout, int32_t ktot) {
  return tc_async_bytes(round_up(cout, 16), round_up(ktot, kTcBK));
}

// Pointwise conv / dense layer out[M, cout] = act(in[M, cin] . W^T + b) on the tcgen05 path; W [w_rows x w_cols]
// (zero beyond: channel padding) given as w_dev[w_rows][w_ld] (w_trans = 0) or as its transpose w_dev[w_cols][w_ld]
// (w_trans = 1: the input-gradient GEMM of the same layer without a host-side transpose).
// The last int of the workspace is the kernel's mbarrier-timeout flag (0 = fine), readable after the stream drains.
YNB_EXPORT int ynb_pwconv_tc_async(const float* in, int32_t in_ld, int32_t in_off, float* out, int32_t out_ld,
                                   int32_t out_off, int32_t out_step, const float* w_dev, int32_t w_ld, int32_t w_rows,
                                   int32_t w_cols, int32_t w_trans, const float* b_dev, int64_t pixels, int32_t cin, int32_t cout, int32_t act,
                                   int32_t mode, void* workspace, int64_t workspace_bytes, void* stream) {
  if (!in || !out || !w_dev || !b_dev || cin % 4 || in_ld % 4 || in_off % 4 || out_ld % 4 || pixels < 1 || cout < 1 ||
      w_cols < 1 || w_cols > cin || w_rows < 1 || w_rows > cout || w_ld < (w_trans ? w_rows : w_cols) ||
      (out_step == 1 && out_off % 4) || cout > 256 || (mode != YNB_GEMM_TC_3XTF32 && mode != YNB_GEMM_TC_TF32))
    return fail(nullptr, YNB_ERR_INVALID, "ynb_pwconv_tc_async: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  TcWeights t;
  t.N = cout; t.Npad = round_up(cout, 16); t.Kpad = round_up(cin, kTcBK);
  AsyncWs a;
  if (!carve_async(workspace, workspace_bytes, t.Npad, t.Kpad, &a))
    return fail(nullptr, YNB_ERR_INVALID, "ynb_pwconv_tc_async: workspace too small or not 256-byte aligned");
  t.hi = a.hi; t.lo = a.lo;
  const int total = t.Npad * t.Kpad;
  pack_tc_weights_kernel<<<(total + 255) / 256, 256, 0, st>>>(w_dev, w_ld, w_rows, w_cols, w_trans, t.hi, t.lo, t.Npad,
                                                              t.Kpad, a.flag);
  TcGemmLaunch L;
  L.w = &t;
  TcGemmParams& p = L.p;
  memset(&p, 0, sizeof(p));
  p.mode = mode; p.num_steps = t.Kpad / kTcBK; p.chunks_per_tap = p.num_steps; p.ksub = (cin + 7) / 8;
  p.M = pixels; p.num_tiles = (pixels + kTcBM - 1) / kTcBM; p.N = cout; p.Npad = t.Npad;
  tc_plan_tmem(p);
  p.a_box_bytes = kTcAStageBytes;
  p.out = out; p.out_ld = out_ld; p.out_off = out_off; p.out_step = out_step;
  p.bias = b_dev; p.act = act; p.err_flag = a.flag;
  p.tma_store = (out_step == 1 && out_off % 4 == 0) ? 1 : 0;
  if (!make_tmap_2d(&t.tm_hi, t.hi, t.Kpad, t.Npad, t.Kpad, t.Npad) ||
      !make_tmap_2d(&t.tm_lo, t.lo, t.Kpad, t.Npad, t.Kpad, t.Npad) ||
      (p.tma_store && !make_tmap_out(&L.tmOut, out + out_off, (uint64_t)round_up(cout, 4), (uint64_t)pixels,
                                     (uint64_t)out_ld)) ||
      !make_tmap_2d(&L.tmA, in + in_off, cin, pixels, in_ld, kTcBM) || !tc_plan_smem(L))
    return fail(nullptr, YNB_ERR_CUDA, "ynb_pwconv_tc_async: tensor map / smem planning failed");
  L.grid = (unsigned)std::min<int64_t>(p.num_tiles, kNumSMs);
  UNIT_TRY(launch_tc_gemm(L, st));
  return YNB_OK;
}

// Dense 3x3 conv, pad 1, stride 1 (w_dev [cout][9][cin] tap-major) — ynb_conv3x3_tc without the host round trip.
YNB_EXPORT int ynb_conv3x3_tc_async(const float* in, int32_t in_ld, float* out, int32_t out_ld, const float* w_dev,
                                    const float* b_dev, int32_t batch, int32_t h, int32_t w_, int32_t cin, int32_t cout,
                                    int32_t act, int32_t mode, void* workspace, int64_t workspace_bytes, void* stream) {
  if (!in || !out || !w_dev || !b_dev || batch <= 0 || h <= 0 || w_ <= 0 || cin <= 0 || cin % kTcBK || in_ld % 4 ||
      out_ld % 4 || cout < 1 || cout > 256 || (mode != YNB_GEMM_TC_3XTF32 && mode != YNB_GEMM_TC_TF32) ||
      (((uintptr_t)in | (uintptr_t)out) & 15u))
    return fail(nullptr, YNB_ERR_INVALID, "ynb_conv3x3_tc_async: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  const int ktot = 9 * cin;
  TcWeights t;
  t.N = cout; t.Npad = round_up(cout, 16); t.Kpad = ktot;
  AsyncWs a;
  if (!carve_async(workspace, workspace_bytes, t.Npad, t.Kpad, &a))
    return fail(nullptr, YNB_ERR_INVALID, "ynb_conv3x3_tc_async: workspace too small or not 256-byte aligned");
  t.hi = a.hi; t.lo = a.lo;
  const int total = t.Npad * t.Kpad;
  pack_tc_weights_kernel<<<(total + 255) / 256, 256, 0, st>>>(w_dev, ktot, cout, ktot, 0, t.hi, t.lo, t.Npad, t.Kpad, a.flag);
  TcGemmLaunch L;
  L.w = &t;
  TcGemmParams& p = L.p;
  memset(&p, 0, sizeof(p));
  p.mode = mode; p.is3x3 = 1;
  p.chunks_per_tap = cin / kTcBK;
  p.num_steps = 9 * p.chunks_per_tap;
  p.H = h; p.W = w_;
  tc_pick_tile(p.H, p.W, &p.TH, &p.TW);
  p.tiles_x = (p.W + p.TW - 1) / p.TW;
  p.tiles_y = (p.H + p.TH - 1) / p.TH;
  p.num_tiles = (int64_t)batch * p.tiles_x * p.tiles_y;
  p.M = (int64_t)batch * h * w_;
  p.N = cout; p.Npad = t.Npad;
  tc_plan_tmem(p);
  p.a_box_bytes = (uint32_t)(p.TH * p.TW * 128);
  p.out = out; p.out_ld = out_ld; p.out_off = 0; p.out_step = 1;
  p.bias = b_dev; p.act = act; p.err_flag = a.flag;
  if (!make_tmap_2d(&t.tm_hi, t.hi, t.Kpad, t.Npad, t.Kpad, t.Npad) ||
      !make_tmap_2d(&t.tm_lo, t.lo, t.Kpad, t.Npad, t.Kpad, t.Npad) ||
      !make_tmap_nhwc(&L.tmA, in, cin, w_, h, batch, in_ld, p.TW, p.TH) || !tc_plan_smem(L))
    return fail(nullptr, YNB_ERR_CUDA, "ynb_conv3x3_tc_async: tensor map / smem planning failed");
  L.grid = (unsigned)std::min<int64_t>(p.num_tiles, kNumSMs);
  UNIT_TRY(launch_tc_gemm(L, st));
  return YNB_OK;
}

// ---- BatchNorm2d in training mode ----------------------------------------------------------------------
namespace {
bool bn_args_ok(long long M, int C, std::initializer_list<int> strides, std::initializer_list<const void*> ptrs) {
  if (M <= 0 || C <= 0 || C % 4) return false;
  for (int v : strides) if (v % 4) return false;
  for (const void* q : ptrs) if (!q || ((uintptr_t)q & 15u)) return false;
  return true;
}
}  // namespace

YNB_EXPORT int64_t ynb_bn_workspace_bytes(int64_t pixels, int32_t channels) {
  return ((int64_t)bn_chunks(pixels) * 2 * channels + 2 * channels) * sizeof(float);
}

YNB_EXPORT int ynb_bn_train_fwd(const float* x, int32_t x_ld, int32_t x_off, float* y, int32_t y_ld, int32_t y_off,
                                const float* gamma, const float* beta, float* running_mean, float* running_var,
                                float* save_mean, float* save_rstd, int64_t pixels, int32_t channels, float eps,
                                float momentum, int32_t act, void* ws, int64_t ws_bytes, void* stream) {
  if (!bn_args_ok(pixels, channels, {x_ld, x_off, y_ld, y_off}, {x, y, gamma, beta, save_mean, save_rstd, ws}) ||
      ws_bytes < ynb_bn_workspace_bytes(pixels, channels) || act < 0 || act > 2)
    return fail(nullptr, YNB_ERR_INVALID, "ynb_bn_train_fwd: bad arguments (channels / strides multiples of 4, 16-byte aligned)");
  cudaStream_t st = (cudaStream_t)stream;
  const int chunks = bn_chunks(pixels);
  const long long rpc = (pixels + chunks - 1) / chunks;
  float* part = (float*)ws;
  float* sums = part + (long long)chunks * 2 * channels;
  dim3 grid(chunks, (channels + kBnCg * 4 - 1) / (kBnCg * 4)), block(kBnCg, kBnSlices);
  bn_colsum_kernel<0><<<grid, block, 0, st>>>(x, x_ld, x_off, nullptr, 0, 0, nullptr, 0, 0, nullptr, nullptr, 0.f, 0, part,
                                              pixels, channels, rpc);
  YNB_COUNT_LAUNCH();
  bn_reduce_finalize_kernel<<<(channels + 31) / 32, dim3(32, kRedSlices), 0, st>>>(part, chunks, pixels, channels, eps, momentum,
                                                                                sums, save_mean, save_rstd, running_mean,
                                                                                running_var);
  YNB_COUNT_LAUNCH();
  const long long total = pixels * (channels / 4);
  const int blocks = (int)std::min<long long>((total + 255) / 256, (long long)kNumSMs * 16);
  bn_apply_kernel<0><<<blocks, 256, 0, st>>>(x, x_ld, x_off, nullptr, 0, 0, nullptr, 0, 0, y, y_ld, y_off, gamma, beta,
                                             save_mean, save_rstd, nullptr, act == YNB_ACT_LEAKY ? 0.1f : 0.0f, act, pixels,
                                             channels);
  YNB_COUNT_LAUNCH();
  UNIT_TRY(cudaGetLastError());
  return YNB_OK;
}

YNB_EXPORT int ynb_bn_train_bwd(const float* dy, int32_t dy_ld, int32_t dy_off, const float* x, int32_t x_ld, int32_t x_off,
                                const float* y, int32_t y_ld, int32_t y_off, const float* gamma, const float* save_mean,
                                const float* save_rstd, float* dx, int32_t dx_ld, int32_t dx_off, float* dgamma_dbeta,
                                int64_t pixels, int32_t channels, int32_t act, void* ws, int64_t ws_bytes, void* stream) {
  if (!bn_args_ok(pixels, channels, {dy_ld, dy_off, x_ld, x_off, dx_ld, dx_off},
                  {dy, x, gamma, save_mean, save_rstd, dx, dgamma_dbeta, ws}) ||
      ws_bytes < ynb_bn_workspace_bytes(pixels, channels) || act < 0 || act > 2 ||
      (act != YNB_ACT_NONE && (!y || y_ld % 4 || y_off % 4)))
    return fail(nullptr, YNB_ERR_INVALID, "ynb_bn_train_bwd: bad arguments (channels / strides multiples of 4, 16-byte aligned)");
  cudaStream_t st = (cudaStream_t)stream;
  const int chunks = bn_chunks(pixels);
  const long long rpc = (pixels + chunks - 1) / chunks;
  float* part = (float*)ws;
  float* sums = part + (long long)chunks * 2 * channels;      // [dbeta | dgamma]
  const float slope = act == YNB_ACT_LEAKY ? 0.1f : 0.0f;
  dim3 grid(chunks, (channels + kBnCg * 4 - 1) / (kBnCg * 4)), block(kBnCg, kBnSlices);
  bn_colsum_kernel<1><<<grid, block, 0, st>>>(x, x_ld, x_off, dy, dy_ld, dy_off, y, y_ld, y_off, save_mean, save_rstd, slope,
                                              act != YNB_ACT_NONE, part, pixels, channels, rpc);
  YNB_COUNT_LAUNCH();
  launch_reduce_partials(part, chunks, 2LL * channels, sums, st);
  const long long total = pixels * (channels / 4);
  const int blocks = (int)std::min<long long>((total + 255) / 256, (long long)kNumSMs * 16);
  bn_apply_kernel<1><<<blocks, 256, 0, st>>>(x, x_ld, x_off, dy, dy_ld, dy_off, y, y_ld, y_off, dx, dx_ld, dx_off, gamma,
                                             nullptr, save_mean, save_rstd, sums, slope, act, pixels, channels);
  YNB_COUNT_LAUNCH();
  UNIT_TRY(cudaMemcpyAsync(dgamma_dbeta, sums + channels, channels * sizeof(float), cudaMemcpyDeviceToDevice, st));
  UNIT_TRY(cudaMemcpyAsync(dgamma_dbeta + channels, sums, channels * sizeof(float), cudaMemcpyDeviceToDevice, st));
  UNIT_TRY(cudaGetLastError());
  return YNB_OK;
}
