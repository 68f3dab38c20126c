// The actor-critic engine: parameter table, packed weights, workspace, and the static kernel
// schedules for forward (Forward module) and forward+loss+backward / clip+Adam (Backward module).
//
// Replaces, behind the same parameter names / shapes / order (so state_dict(), nn2redis blobs and
// .pt checkpoints stay interchangeable, nn/base.py:60-81):
//   AtariPreNet   USTC_lab/nn/atari_encoder.py:11-32     NavPreNet / NavPedPreNet  nn/nav_encoder.py:12-79
//   NavPreNet1D   nn/nav_encoder.py:82-128               MLPPreNet                 nn/mlp_encoder.py:12-29
//   CategoricalActor / GaussionActor nn/actor.py:43-101  Critic nn/critic.py:6-21
//   PPO.forward / PPO.learn          nn/ppo.py:72-142    (tower sharing per runner/utils.py:59-170)
//
// Design (B200-first, not a port of autograd): no graph is recorded.  Each encoder family is a
// fixed schedule of GEMMs (convolutions as im2col GEMMs over NHWC activations) plus streaming glue
// kernels, run over micro-batches that keep the working set bounded; weight gradients accumulate
// across micro-batches directly in the flat gradient buffer (or its packed twin), which is what the
// data-parallel learner all-reduces in one NCCL call before the fused clip+Adam.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <string>
#include <unordered_map>
#include <vector>

#include "common.cuh"
#include "layer_ops.h"
#include "prep_kernels.cuh"

namespace ddrl {

struct TensorInfo {
  std::string name;
  int64_t shape[4];
  int ndim;
  int64_t offset, numel;
};

// One GEMM layer y[M,N] = act(x[M,K] W[N,K]^T + b): a Linear, or a Conv over its im2col matrix.
struct Lin {
  int N = 0, K = 0, ldw = 0;
  int w_t = -1, b_t = -1;        // tensor-table indices
  int I = 1, J = 0;              // packed[o, i*J + j] = ref[o, j*I + i]
  bool packed = false;
  int act = 0;
  float* wp = nullptr;           // packed weight [N, ldw]   (when packed)
  float *wp_hi = nullptr, *wp_lo = nullptr;   // its tf32 hi / lo split (tc2 engine), refreshed with wp
  W16 w16;                       // scaled fp16 split (+ transposed twin) of wp (tc3 engine), refreshed with wp
  float* dwp = nullptr;          // packed weight gradient   (when packed and training)
  int s2d_s = 0, s2d_C = 0, s2d_KH = 0, s2d_KW = 0;   // space-to-depth first layer: packing follows pack_weight_s2d
  bool s2d_fwd_only = false;     // ... for the forward weights only: the weight gradient runs on the im2col matrix (k = c,kh,kw)
  int seg = 0;                   // backward segment after which this layer's gradient is final (assign_segments)
};

struct Arena {
  char* base = nullptr;
  size_t cap = 0, used = 0;
  float* take(size_t nfloats) {
    const size_t bytes = (nfloats * sizeof(float) + 255) & ~size_t(255);
    if (used + bytes > cap) return nullptr;
    float* p = reinterpret_cast<float*>(base + used);
    used += bytes;
    return p;
  }
};

enum { ACT_NONE = 0, ACT_RELU = 1, ACT_LEAKY = 2 };

struct Tower {
  int arch = 0, in_ch = 0, feat = 512;
  std::string prefix;
  std::vector<Lin> L;            // layer order is arch specific (see build_tower)
  ConvGeom g[5];                 // conv geometries (arch specific slots)
  bool implicit[5] = {false, false, false, false, false};   // layer runs on the implicit-GEMM (tap-TMA) path
  int conv_lin[5] = {-1, -1, -1, -1, -1};                   // index into L of the conv in slot g[i]
  std::vector<DgradClass> dg[5];                            // data-gradient parity classes (+ packed weights)
  DgradFused df[5] = {};                                    // tc2: all classes of a strided layer as one GEMM
  // cross-tower fusion of the first conv (unshared towers read the same observation): 0 none, 1 owner of the shared
  // im2col / a1 / da1 buffers (tower 0), 2 borrower.  conv slot 1 then reads channels [in1_coff, +C) of a in1_ctot-wide tensor.
  int fuse_role = 0, in1_ctot = 0, in1_coff = 0;
  bool s2d0 = false;                                        // conv slot 0 runs on the space-to-depth observation
  bool s2d_infer = false;                                   // fused first conv: inference runs on the s2d observation
  bool s2d_train = false;                                   // ... and so does training (tc3 engine): no im2col matrix at all
  bool borrow_cols = false;                                 // second unshared tower: the observation-side im2col matrices are tower 0's
  ConvGeom gs = {};                                         // its stride-1 NHWC geometry (buf[0] holds the s2d tensor)
  // per-micro-batch buffers
  std::vector<float*> buf;
  std::vector<uint8_t*> idx;
  float* h = nullptr;            // encoder output [MB, feat]
  float* dh = nullptr;           // its gradient
};

}  // namespace ddrl

using namespace ddrl;

struct ddrl_net {
  ddrl_net_desc d;
  std::vector<TensorInfo> T;
  int64_t P = 0;
  float *params = nullptr, *grads = nullptr, *am = nullptr, *av = nullptr;
  bool dirty = true;             // packed weights stale
  std::vector<Tower> towers;     // shared: [prenet]; unshared: [actor.pre, critic.pre]
  int t_aw = -1, t_ab = -1, t_cw = -1, t_cb = -1, t_logstd = -1;
  int ldA = 0;                   // padded row stride of the actor head output
  // workspace
  Arena ws;
  int MB = 0;                    // micro-batch rows the workspace is sized for
  bool ws_train = false;
  float *logits = nullptr, *vout = nullptr, *dlogits = nullptr, *dv = nullptr, *stage = nullptr;
  // extra value heads on the critic-side feature (nn/ppo.py:63-64 add_critic; share-CNN mode): parameters and gradients
  // live OUTSIDE the flat buffers (the reference's optimisers are built before add_critic and never see them)
  struct ExtraCritic { const float *w, *b; float *dw, *db; int in_loss; };
  std::vector<ExtraCritic> extra;
  float *vout_x = nullptr, *dv_x = nullptr;    // [kMaxExtra, MB]
  char* packed_base = nullptr;   // packed weights + packed grads arena
  char* split_base = nullptr;    // tc2 engine: [hi mirror of the packed arena | lo mirror]
  size_t packed_bytes = 0, packed_grad_off = 0, packed_grad_bytes = 0;
  int64_t seg_begin[3];
  int nseg = 1;
  bool fuse0 = false;            // both towers' first conv as ONE GEMM over the shared im2col matrix (N = 2 x Cout)
  // ... and, in the Forward module (no training workspace), as an implicit stride-1 conv over the space-to-depth
  // observation: no im2col matrix at all (3.4 GB per 8192 rows, 1.9 ms to build).  Measured (profiles/r1f_*): Forward
  // 2.16 -> 2.38 M actions/s; in the learner the im2col matrix is cached across the 10 iterations and needed by the weight
  // gradient anyway, and the im2col GEMM (842 us) beats the implicit kernel (944 us), so training keeps it.
  bool fuse_s2d = false;
  // tc3 engine: the learner runs the fused first conv (forward AND weight gradient) on the space-to-depth observation too --
  // the 3.4 GB im2col matrix and its two HBM-bound passes per iteration are gone (DDRL_NO_S2D_TRAIN=1 keeps the im2col GEMM)
  bool s2d_train = false;
  float* s2dbuf = nullptr;       // [MB, H/s, W/s, s*s*C] space-to-depth observation of the micro-batch
  // ... and its fp16 split (tc3 engine, DDRL_NO_PRESPLIT=1 turns it off): planes hi [MB, ...] | lo' [MB, ...], written once per
  // staged micro-batch by tc3_presplit.  The first conv and its weight gradient (20 launches per learn call on the same
  // observation) then take both MMA operands straight from TMA: no per-use split, no splitter warps in those launches.
  void* s2d16 = nullptr;
  size_t s2d16_plane = 0;        // bytes per plane
  // activation buffers with a registered sign-bit tensor (tc3 engine, NatureCNN towers: the conv outputs whose leaky'
  // the data gradients of the next layer need) -- see tc3_signbits_register
  std::vector<const float*> signbit_bases;
  float* w0s2d = nullptr;        // [2 x Cout, K] both towers' conv1 weights in the space-to-depth K order (packed arena)
  float* bias0c = nullptr;       // its concatenated bias [2 x Cout]
  // observation-side im2col matrices in the workspace belong to (obs pointer, rows) of the last single-chunk backward
  const float* cols_obs0 = nullptr;
  int cols_rows = -1;
  // ---- tc3 engine: scaled fp16 weight operands and the amax scalars of every GEMM operand
  char* h16_base = nullptr;      // fp16 arena of the split weights
  size_t h16_bytes = 0;
  float* amax_dev = nullptr;     // [kAmaxSlots] device scalars: [0, kAmaxWeights) weights (persistent), the rest activations
  int amax_w_used = 0, amax_a_used = 0;
  struct SplitJob { const float* w; int rows, K, ldw; W16* dst; bool transposed; };
  std::vector<SplitJob> split_jobs;                 // every weight operand, in repack order
  std::vector<W16> w16_extra;                       // operands that are not a Lin / dgrad class (fused first conv, s2d weights)
  std::unordered_map<const float*, const W16*> w16_of;   // packed fp32 operand -> its split
  struct AmaxEntry { int slot; unsigned long long epoch; bool persistent; };
  std::unordered_map<std::string, AmaxEntry> amax_keys;  // activation view -> slot (valid while epoch == amax_epoch)
  unsigned long long amax_epoch = 1;
  W16 w16_fuse0, w16_s2d;
  // the weight preparation after every optimiser step is ~90 tiny independent launches: they are spread round-robin over
  // side streams (fork / join with events) so their launch latencies overlap instead of adding up
  // ---- CUDA graphs of the steady-state learn iteration (iterations 2..10 of PPO.learn run the SAME launches on the SAME
  // pointers): the backward pass and the optimiser step + weight re-preparation are captured once per argument set and
  // replayed with one cudaGraphLaunch each (DDRL_NO_GRAPH=1: every launch goes to the stream, as the profiler hooks need)
  struct GraphEntry {
    std::string key;
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    cudaGraphNode_t adam_node = nullptr;
    long long launches = 0;
    unsigned long long used = 0;
    // a body with segment cuts (the backward pass) is a CHAIN of graphs: pre[0], pre[1], ..., then `exec`
    std::vector<cudaGraph_t> pre_graphs;
    std::vector<cudaGraphExec_t> pre_execs;
    std::vector<long long> pre_launches;
  };
  // segment cuts of the backward pass (seg_cut): while a capture is running each cut closes the current graph and opens the
  // next, so that a data-parallel learner can hand the gradients that are final after segment k to NCCL while segment k + 1
  // runs (nn/ppo.py learn).  Outside a capture a cut does nothing and the pass ends with ONE un-permutation of everything.
  struct Capture {
    bool active = false, failed = false;
    int seg = 0;
    long long l0 = 0;
    std::vector<cudaGraph_t> done;
    std::vector<long long> launches;
  } cap;
  int n_bwd_seg = 1;               // segments of a captured backward pass (towers + 1)
  std::vector<GraphEntry> graphs;
  unsigned long long graph_clock = 0;
  cudaStream_t cap_stream = nullptr;
  bool graphs_off = false;
  // minibatch passes (ddrl_net_backward_minibatch): a failed capture turns off only these graphs; a key runs on the stream
  // the first time it is seen (that call performs the one-time allocations a capture must not contain)
  bool mb_graphs_off = false;
  std::vector<std::string> mb_seen;
  double* sumsq_dev = nullptr;     // clip+Adam norm scratch of THIS net
  // weight preparation as three dependent multi-job launches (prep.cu): [re-packs + amax-slot zeroing] -> [amax + tf32
  // mirrors] -> [fp16 splits]; and the gradient un-permutation that ends a backward pass as one more
  PrepTable prep[3], unprep;
  std::vector<PrepTable> unprep_seg;   // the gradient un-permutation split by backward segment
  bool prep_ready = false;
  static constexpr int kSide = 8;
  cudaStream_t side[kSide] = {};
  cudaEvent_t ev_fork = nullptr, ev_join[kSide] = {};
  bool amax_persist_next = false;  // the next gemm()'s activation operand is observation-side staging (persistent amax entry)
};

namespace ddrl {

constexpr int kAmaxSlots = 1024, kAmaxWeights = 256;
constexpr int kMaxExtra = 2;      // extra critic heads ("suppose 3 critic net at most", nn/ppo.py:93)
// mode 3 (tc3) is a superset of mode 2: same lowering decisions; the tc2 kernels keep the launches tc3 does not take
static inline bool tc3_mode(const ddrl_net* n) { return n->d.gemm_mode == DDRL_GEMM_TC3_F16; }
// NavPreNet1D: channels of the laser observation [B, laser_ch, 960].  The reference's encoder takes 1 (nn/nav_encoder.py:87);
// 3 is the NON-reference "3 x 960" variant SURVEY 8(d) asks to bench (3-frame laser stacking is an env option only)
static inline int laser_ch_of(const ddrl_net* n) { return n->d.laser_ch > 0 ? n->d.laser_ch : 1; }
static inline bool tc_mode(const ddrl_net* n) { return n->d.gemm_mode == DDRL_GEMM_TC_3XTF32 || n->d.gemm_mode == DDRL_GEMM_TC2_TMEM || tc3_mode(n); }
static inline bool tc2_mode(const ddrl_net* n) { return n->d.gemm_mode == DDRL_GEMM_TC2_TMEM || tc3_mode(n); }

static void graphs_clear(ddrl_net* n);

// The tc3 weight gradient sums the dy columns (bias gradient) while its epilogue warps convert the dy tiles: those warps are
// idle 90 % of the kernel, so the separate column-sum pass over dy (5.8 % of a Pong step) disappears.  (While the
// conversion lived in the splitter warps -- that kernel's critical role -- the fused sums cost what they saved, profiles/r2h_*.)
// DDRL_TC3_FUSE_COLSUM=0 brings the separate pass back.
static inline bool fuse_colsum() {
  static const bool on = [] { const char* e = getenv("DDRL_TC3_FUSE_COLSUM"); return !(e && e[0] == '0'); }();
  return on;
}

// ---- amax registry of the tc3 engine -------------------------------------------------------------------------------
// A view is (pointer, rows, cols, row stride); contiguous views are keyed by (pointer, element count) so that a conv
// output [B*Ho*Wo, C] and the next layer's [B, Ho*Wo*C] read of it are the same key.  Only EXACT matches are trusted:
// any other view of a buffer gets its own standalone reduction.  Slots of the activation region are zeroed at the start
// of every engine pass; producers atomicMax into them, so a slot written several times in one pass (micro-batches,
// shared scratch buffers) holds an upper bound -- which is all the scale needs.
static std::string amax_key(const float* p, long long rows, long long cols, long long ld) {
  char b[96];
  if (ld == cols) snprintf(b, sizeof(b), "%p:%lld", (const void*)p, rows * cols);
  else snprintf(b, sizeof(b), "%p:%lld:%lld:%lld", (const void*)p, rows, cols, ld);
  return b;
}
static void amax_new_pass(ddrl_net* n, cudaStream_t s, bool keep_persistent) {
  if (!n->amax_dev) return;
  ++n->amax_epoch;
  if (!keep_persistent)
    for (auto& kv : n->amax_keys) if (kv.second.persistent) kv.second.epoch = 0;
  cudaMemsetAsync(n->amax_dev + kAmaxWeights, 0, sizeof(float) * (kAmaxSlots - kAmaxWeights), s);
}
// persistent entries (observation-side staging that survives the iterations of one learn call) live in the weight region,
// which the per-pass memset does not touch
static int amax_slot_index(ddrl_net* n, const std::string& key, bool persistent = false) {
  auto it = n->amax_keys.find(key);
  if (it != n->amax_keys.end()) return it->second.slot;
  int slot;
  if (persistent) {
    if (n->amax_w_used >= kAmaxWeights) return -1;
    slot = n->amax_w_used++;
  } else {
    if (n->amax_a_used >= kAmaxSlots - kAmaxWeights) return -1;
    slot = kAmaxWeights + n->amax_a_used++;
  }
  n->amax_keys[key] = {slot, 0, persistent};
  return slot;
}
// slot a tc3 epilogue accumulates the amax of its output into (nullptr: not tracked)
static float* amax_out_slot(ddrl_net* n, const float* p, long long rows, long long cols, long long ld) {
  if (!tc3_mode(n) || !n->amax_dev) return nullptr;
  const std::string key = amax_key(p, rows, cols, ld);
  const int slot = amax_slot_index(n, key);
  if (slot < 0) return nullptr;
  n->amax_keys[key].epoch = n->amax_epoch;
  return n->amax_dev + slot;
}
// amax of an operand view: the producer's slot when this exact view was written by a tracked producer in this pass,
// otherwise a standalone reduction (result cached for the rest of the pass)
static int amax_in_slot(ddrl_net* n, const float* p, long long rows, long long cols, long long ld, cudaStream_t s, const float** out,
                        bool persistent = false) {
  const std::string key = amax_key(p, rows, cols, ld);
  const int slot = amax_slot_index(n, key, persistent);
  if (slot < 0) return DDRL_E_STATE;
  ddrl_net::AmaxEntry& e = n->amax_keys[key];
  *out = n->amax_dev + slot;
  if (e.persistent ? e.epoch != 0 : e.epoch == n->amax_epoch) return DDRL_OK;
  e.epoch = n->amax_epoch;
  return amax_f32(p, rows, (int)cols, ld, n->amax_dev + slot, e.persistent, s);
}
// hi / lo mirrors of a pointer into the packed arena
static inline const float* hi_of(const ddrl_net* n, const float* p) {
  return reinterpret_cast<const float*>(n->split_base + (reinterpret_cast<const char*>(p) - n->packed_base));
}
static inline const float* lo_of(const ddrl_net* n, const float* p) {
  return reinterpret_cast<const float*>(n->split_base + n->packed_bytes + (reinterpret_cast<const char*>(p) - n->packed_base));
}
static inline bool in_packed(const ddrl_net* n, const float* p) {
  const char* c = reinterpret_cast<const char*>(p);
  return n->packed_base && c >= n->packed_base && c < n->packed_base + n->packed_bytes;
}

static int find_tensor(const ddrl_net* n, const std::string& name) {
  for (size_t i = 0; i < n->T.size(); ++i)
    if (n->T[i].name == name) return (int)i;
  return -1;
}

static void add_tensor(ddrl_net* n, const std::string& name, std::initializer_list<int64_t> shape) {
  TensorInfo t;
  t.name = name;
  t.ndim = (int)shape.size();
  t.numel = 1;
  int i = 0;
  for (auto s : shape) { t.shape[i++] = s; t.numel *= s; }
  for (; i < 4; ++i) t.shape[i] = 1;
  t.offset = n->P;
  n->P += t.numel;
  n->T.push_back(t);
}

// reference named_parameters() order of one encoder (SURVEY App. C)
static void add_encoder_tensors(ddrl_net* n, const std::string& pre, int arch, int in_ch, int feat) {
  auto conv = [&](const char* nm, int o, int c, int kh, int kw) {
    add_tensor(n, pre + nm + ".weight", {o, c, kh, kw});
    add_tensor(n, pre + nm + ".bias", {o});
  };
  auto lin = [&](const char* nm, int o, int i) {
    add_tensor(n, pre + nm + ".weight", {o, i});
    add_tensor(n, pre + nm + ".bias", {o});
  };
  switch (arch) {
    case DDRL_ARCH_ATARI:
      conv("conv1", 32, in_ch, 8, 8); conv("conv2", 64, 32, 4, 4); conv("conv3", 64, 64, 3, 3); lin("linear", 512, 3136);
      break;
    case DDRL_ARCH_NAV:
    case DDRL_ARCH_NAVPED:
      conv("conv1", 64, in_ch, 3, 3); conv("conv2", 128, 64, 3, 3); conv("conv3", 256, 128, 3, 3);
      lin("fc0.0", 512, 9216); lin("fc1.0", 512, 521); lin("fc2", 512, 512);
      break;
    case DDRL_ARCH_NAV1D:
      conv("conv1", 64, in_ch, 7, 7); conv("conv2", 128, 64, 5, 5); conv("conv3", 256, 128, 3, 3);
      add_tensor(n, pre + "conv1d1.weight", {32, laser_ch_of(n), 5}); add_tensor(n, pre + "conv1d1.bias", {32});
      add_tensor(n, pre + "conv1d2.weight", {32, 32, 3}); add_tensor(n, pre + "conv1d2.bias", {32});
      lin("fc_1d.0", 256, 7616); lin("fc0.0", 512, 6400); lin("fc1.0", 512, 773); lin("fc2", 512, 512);
      break;
    case DDRL_ARCH_MLP:
      lin("fc0.0", feat, in_ch);
      break;
  }
}

static int round4(int x) { return (x + 3) & ~3; }

static Lin make_lin(ddrl_net* n, const std::string& wname, int N, int K, int I, int J, int act) {
  Lin l;
  l.N = N; l.K = K; l.I = I; l.J = J; l.act = act;
  l.ldw = round4(K);
  // always keep an engine-side copy: besides the layout change it guarantees the 16-byte alignment TMA needs
  // (flat-buffer offsets of e.g. critic.pre.* are odd because of the [A,512]+[A]+[1,512]+[1] head tensors)
  l.packed = true;
  l.w_t = find_tensor(n, wname + ".weight");
  l.b_t = find_tensor(n, wname + ".bias");
  return l;
}

static ConvGeom conv_geom(int H, int W, int C, bool nchw, int KH, int KW, int stride, int pad) {
  ConvGeom g;
  g.H = H; g.W = W; g.C = C;
  if (nchw) { g.sc = (long long)H * W; g.sh = W; g.sw = 1; g.sb = (long long)C * H * W; g.order = 1; }
  else { g.sc = 1; g.sw = C; g.sh = (long long)W * C; g.sb = (long long)H * W * C; g.order = 0; }
  g.KH = KH; g.KW = KW; g.stride = stride; g.pad = pad;
  g.Ho = (H + 2 * pad - KH) / stride + 1;
  g.Wo = (W + 2 * pad - KW) / stride + 1;
  g.K = C * KH * KW;
  g.ldc = round4(g.K);
  return g;
}

static void build_tower(ddrl_net* n, Tower& t, const std::string& prefix, int arch, int in_ch, int feat) {
  t.arch = arch; t.in_ch = in_ch; t.feat = feat; t.prefix = prefix;
  auto P = [&](const char* s) { return prefix + s; };
  switch (arch) {
    case DDRL_ARCH_ATARI:
      t.g[0] = conv_geom(84, 84, in_ch, true, 8, 8, 4, 0);       // -> 20x20x32
      t.g[1] = conv_geom(20, 20, 32, false, 4, 4, 2, 0);         // -> 9x9x64
      t.g[2] = conv_geom(9, 9, 64, false, 3, 3, 1, 0);           // -> 7x7x64
      t.L.push_back(make_lin(n, P("conv1"), 32, t.g[0].K, 1, t.g[0].K, ACT_LEAKY));
      t.L.push_back(make_lin(n, P("conv2"), 64, t.g[1].K, 16, 32, ACT_LEAKY));
      t.L.push_back(make_lin(n, P("conv3"), 64, t.g[2].K, 9, 64, ACT_LEAKY));
      t.L.push_back(make_lin(n, P("linear"), 512, 3136, 49, 64, ACT_NONE));
      break;
    case DDRL_ARCH_NAV:
    case DDRL_ARCH_NAVPED:
      t.g[0] = conv_geom(48, 48, in_ch, true, 3, 3, 1, 1);       // -> 48x48x64 -> pool 24
      t.g[1] = conv_geom(24, 24, 64, false, 3, 3, 1, 1);         // -> 24x24x128 -> pool 12
      t.g[2] = conv_geom(12, 12, 128, false, 3, 3, 1, 1);        // -> 12x12x256 -> pool 6
      t.L.push_back(make_lin(n, P("conv1"), 64, t.g[0].K, 1, t.g[0].K, ACT_RELU));
      t.L.push_back(make_lin(n, P("conv2"), 128, t.g[1].K, 9, 64, ACT_RELU));
      t.L.push_back(make_lin(n, P("conv3"), 256, t.g[2].K, 9, 128, ACT_RELU));
      t.L.push_back(make_lin(n, P("fc0.0"), 512, 9216, 36, 256, ACT_RELU));
      t.L.push_back(make_lin(n, P("fc1.0"), 512, 521, 1, 521, ACT_RELU));
      t.L.push_back(make_lin(n, P("fc2"), 512, 512, 1, 512, ACT_NONE));
      break;
    case DDRL_ARCH_NAV1D:
      t.g[0] = conv_geom(48, 48, in_ch, true, 7, 7, 1, 1);       // -> 44x44x64 -> pool 22
      t.g[1] = conv_geom(22, 22, 64, false, 5, 5, 1, 1);         // -> 20x20x128 -> pool 10
      t.g[2] = conv_geom(10, 10, 128, false, 3, 3, 1, 1);        // -> 10x10x256 -> pool 5
      t.g[3] = conv_geom(1, 960, laser_ch_of(n), true, 1, 5, 2, 0);   // laser conv1d1 -> 478 x 32 (laser_ch = 1 in the reference)
      t.g[4] = conv_geom(1, 478, 32, false, 1, 3, 2, 0);         // laser conv1d2 -> 238 x 32
      t.L.push_back(make_lin(n, P("conv1"), 64, t.g[0].K, 1, t.g[0].K, ACT_RELU));
      t.L.push_back(make_lin(n, P("conv2"), 128, t.g[1].K, 25, 64, ACT_RELU));
      t.L.push_back(make_lin(n, P("conv3"), 256, t.g[2].K, 9, 128, ACT_RELU));
      t.L.push_back(make_lin(n, P("conv1d1"), 32, t.g[3].K, 1, t.g[3].K, ACT_NONE));
      t.L.push_back(make_lin(n, P("conv1d2"), 32, 96, 3, 32, ACT_NONE));
      t.L.push_back(make_lin(n, P("fc_1d.0"), 256, 7616, 238, 32, ACT_RELU));
      t.L.push_back(make_lin(n, P("fc0.0"), 512, 6400, 25, 256, ACT_RELU));
      t.L.push_back(make_lin(n, P("fc1.0"), 512, 773, 1, 773, ACT_RELU));
      t.L.push_back(make_lin(n, P("fc2"), 512, 512, 1, 512, ACT_NONE));
      break;
    case DDRL_ARCH_MLP:
      t.L.push_back(make_lin(n, P("fc0.0"), feat, in_ch, 1, in_ch, ACT_RELU));
      break;
  }
  // conv slot -> layer index; inner convs (NHWC input, channel count a multiple of 32) take the implicit-GEMM path
  const int nconv = arch == DDRL_ARCH_ATARI ? 3 : (arch == DDRL_ARCH_NAV1D ? 5 : (arch == DDRL_ARCH_MLP ? 0 : 3));
  const char* no_implicit = getenv("DDRL_NO_IMPLICIT");
  for (int i = 0; i < nconv; ++i) {
    t.conv_lin[i] = i;
    const ConvGeom& g = t.g[i];
    const int Cout = t.L[i].N;
    if (!tc_mode(n) || g.order != 0 || g.C % 32 != 0 || Cout % 32 != 0) continue;
    if (no_implicit && no_implicit[0] == '1') continue;
    static const float* const kAligned = reinterpret_cast<const float*>(uintptr_t(256));
    ConvOp o = conv_op_fwd(g, kAligned, g.C, 0, 1);
    if (!conv_tc_supported(o, false) || !conv_tc_supported(o, true)) continue;
    std::vector<DgradClass> cls;
    if (conv_dgrad_plan(g, Cout, cls) != DDRL_OK) continue;
    if (!conv_dgrad_supported(g, Cout, cls, kAligned, Cout, 0, 1)) continue;
    t.implicit[i] = true;
    t.dg[i] = cls;
    if (tc2_mode(n) && g.stride > 1) conv_dgrad_fused_plan(g, Cout, t.df[i]);    // leaves df.on = false if unsupported
    if (t.df[i].on) t.dg[i].clear();                 // the per-class repacks would never be read
  }
  // first layer on the raw NCHW observation: a strided valid conv whose extents divide by the stride becomes a stride-1
  // implicit conv over the space-to-depth tensor (same size as the observation; no im2col matrix)
  // Measured on B200 (profiles/r1c_tc2_experiments.md): with N = 32 the implicit kernels are bound by per-tile / per-K-block
  // pipeline cost, not by HBM, and the 78 %-filled 6x20-pixel tiles make conv1 forward 822 us vs 596 us on the cached im2col
  // matrix -- so this path is opt-in (DDRL_S2D=1) until the N = 32 tile cost drops.
  const char* use_s2d = getenv("DDRL_S2D");
  if (nconv > 0 && tc_mode(n) && !(no_implicit && no_implicit[0] == '1') && use_s2d && use_s2d[0] == '1') {
    const ConvGeom& g = t.g[0];
    const int st = g.stride, Cout = t.L[0].N;
    if (g.order == 1 && g.sw == 1 && g.pad == 0 && st > 1 && g.KH % st == 0 && g.KW % st == 0 && g.H % st == 0 &&
        g.W % st == 0 && (st * st * g.C) % 32 == 0 && Cout % 32 == 0 && (size_t)g.C * st * g.W * 4 <= 48 * 1024) {
      ConvGeom gs = conv_geom(g.H / st, g.W / st, st * st * g.C, false, g.KH / st, g.KW / st, 1, 0);
      static const float* const kAligned = reinterpret_cast<const float*>(uintptr_t(256));
      ConvOp o = conv_op_fwd(gs, kAligned, gs.C, 0, 1);
      if (gs.Ho == g.Ho && gs.Wo == g.Wo && gs.K == g.K && conv_tc_supported(o, false) && conv_tc_supported(o, true)) {
        t.s2d0 = true;
        t.gs = gs;
        Lin& l = t.L[0];
        l.s2d_s = st; l.s2d_C = g.C; l.s2d_KH = g.KH; l.s2d_KW = g.KW;
      }
    }
  }
}

// ---- engine dispatch ------------------------------------------------------------------
// act 3 / 4: C = (A op B) * relu' / leaky' of mask (same shape and row stride as C)
static int gemm(const ddrl_net* n, int form, int M, int N, int K, const float* A, int lda, const float* B, int ldb,
                float* C, int ldc, const float* bias, int act, int beta, int trans_c, cudaStream_t s,
                const float* mask = nullptr) {
  // tc3: forward / dgrad GEMMs whose B operand is a packed weight with a scaled-fp16 split (form 1 reads the transposed twin)
  if (tc3_mode(n) && form != 2 && !beta && !trans_c) {
    auto it = n->w16_of.find(B);
    if (it != n->w16_of.end()) {
      const W16& w = *it->second;
      const void *hi = form == 0 ? w.hi : w.hiT, *lo = form == 0 ? w.lo : w.loT;
      const int ld16 = form == 0 ? w.ld : w.ldT;
      if (hi && tc3_gemm_supported(M, N, K, A, lda, hi, lo, ld16)) {
        ddrl_net* nn = const_cast<ddrl_net*>(n);
        const float* ama = nullptr;
        const bool persist = nn->amax_persist_next;
        nn->amax_persist_next = false;
        int r = amax_in_slot(nn, A, M, K, lda, s, &ama, persist);
        if (r != DDRL_OK) return r;
        return tc3_gemm(M, N, K, A, lda, hi, lo, ld16, ama, w.amax, C, ldc, bias, act, mask, amax_out_slot(nn, C, M, N, ldc), s);
      }
    }
  }
  const_cast<ddrl_net*>(n)->amax_persist_next = false;
  // tc2: forward / dgrad GEMMs whose B operand is a packed weight (pre-split mirrors exist)
  if (tc2_mode(n) && form != 2 && !beta && !trans_c && in_packed(n, B) &&
      tc2_gemm_supported(form, M, N, K, A, lda, hi_of(n, B), lo_of(n, B), ldb))
    return tc2_gemm(form, M, N, K, A, lda, hi_of(n, B), lo_of(n, B), ldb, C, ldc, bias, act, mask, s);
  if (tc_mode(n) && gemm_tc_supported(form, M, N, K, A, lda, B, ldb, C, ldc, trans_c))
    return gemm_tc(form, M, N, K, A, lda, B, ldb, C, ldc, bias, act, beta, trans_c, s, mask);
  if (act >= 3) {
    int r = gemm_simt(form, M, N, K, A, lda, B, ldb, C, ldc, bias, 0, beta, trans_c, s);
    if (r != DDRL_OK) return r;
    return act_bwd(C, ldc, mask, ldc, M, N, act - 2, s);
  }
  return gemm_simt(form, M, N, K, A, lda, B, ldb, C, ldc, bias, act, beta, trans_c, s);
}

static const float* W_of(const ddrl_net* n, const Lin& l) { return l.packed ? l.wp : n->params + n->T[l.w_t].offset; }
static float* dW_of(const ddrl_net* n, const Lin& l) { return l.packed ? l.dwp : n->grads + n->T[l.w_t].offset; }
static const float* b_of(const ddrl_net* n, const Lin& l) { return n->params + n->T[l.b_t].offset; }
static float* db_of(const ddrl_net* n, const Lin& l) { return n->grads + n->T[l.b_t].offset; }

#define TRY(x)                \
  do {                        \
    int _r = (x);             \
    if (_r != DDRL_OK) return _r; \
  } while (0)

// y = act(x W^T + b)
static int lin_fwd(const ddrl_net* n, const Lin& l, const float* x, int ldx, float* y, int ldy, long long M, cudaStream_t s) {
  ddrl_net* nn = const_cast<ddrl_net*>(n);
  const bool persist = nn->amax_persist_next;          // set by the caller when x is observation-side staging
  nn->amax_persist_next = false;
  if (l.K <= 36 && l.act <= 2 && thin_supported(M, l.N, l.K, x, ldx, y, ldy))
    return thin_fwd(x, ldx, W_of(n, l), l.ldw, b_of(n, l), y, M, l.N, l.K, l.act, s);
  nn->amax_persist_next = persist;
  return gemm(n, 0, (int)M, l.N, l.K, x, ldx, W_of(n, l), l.ldw, y, ldy, b_of(n, l), l.act, 0, 0, s);
}
// dy holds dL/d(pre-activation) of this layer (the activation derivative was applied by whoever produced dy).
// db += colsum(dy); dW += dy^T x; dx = (dy W) * act'(mask)   (ncols_dx: leading columns of dx wanted;
// mask_act: 0 none, 1 relu, 2 leaky -- the activation that produced x, i.e. of the layer BELOW; mask = that x)
static int lin_bwd(const ddrl_net* n, const Lin& l, const float* x, int ldx, float* dy, int ldy, float* dx, int lddx,
                   int ncols_dx, int mask_act, const float* mask, long long M, cudaStream_t s) {
  ddrl_net* nn = const_cast<ddrl_net*>(n);
  const bool persist = nn->amax_persist_next;          // set by the caller when x is observation-side staging
  nn->amax_persist_next = false;
  // dW[N, K] += dy[M,N]^T x[M,K]
  const bool al = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dy)) & 15) == 0 && ldx % 4 == 0 && ldy % 4 == 0;
  const bool thin = l.K <= 36 && thin_supported(M, l.N, l.K, x, ldx, dy, ldy);
  const bool w3 = !thin && tc3_mode(n) && al && l.K >= 32 && !getenv("DDRL_TC3_NO_WGRAD");
  const bool fuse_cs = fuse_colsum();
  if (!(w3 && fuse_cs)) TRY(colsum_add(dy, ldy, M, l.N, db_of(n, l), s));
  if (thin)
    TRY(thin_wgrad(x, ldx, dy, dW_of(n, l), l.ldw, M, l.N, l.K, s));
  else if (w3) {
    const float *amx = nullptr, *amy = nullptr;
    TRY(amax_in_slot(nn, x, M, l.K, ldx, s, &amx, persist));
    TRY(amax_in_slot(nn, dy, M, l.N, ldy, s, &amy));
    TRY(tc3_wgrad(l.K, l.N, M, x, ldx, dy, ldy, amx, amy, dW_of(n, l), l.ldw, s, fuse_cs ? db_of(n, l) : nullptr));
  }
  else if (tc2_mode(n) && al && l.K >= 32)
    TRY(tc2_wgrad(l.K, l.N, M, x, ldx, dy, ldy, dW_of(n, l), l.ldw, s));
  // older engines: run with the larger of (N, K) on the 128-row side
  else if (l.N >= 128 || l.N >= l.K)
    TRY(gemm(n, 2, l.N, l.K, (int)M, dy, ldy, x, ldx, dW_of(n, l), l.ldw, nullptr, 0, 1, 0, s));
  else
    TRY(gemm(n, 2, l.K, l.N, (int)M, x, ldx, dy, ldy, dW_of(n, l), l.ldw, nullptr, 0, 1, 1, s));
  if (dx) TRY(gemm(n, 1, (int)M, ncols_dx, l.N, dy, ldy, W_of(n, l), l.ldw, dx, lddx, nullptr, mask_act ? mask_act + 2 : 0, 0, 0, s,
                   mask_act ? mask : nullptr));
  return DDRL_OK;
}

// ---- workspace ------------------------------------------------------------------------
// per-sample float counts of a tower's buffers, in the order tower_alloc() carves them
static void tower_sizes(const Tower& t, bool train, std::vector<size_t>& f, std::vector<size_t>& u8) {
  auto cols = [&](const ConvGeom& g) {
    const int gi = (int)(&g - &t.g[0]);
    if (gi == 0 && t.s2d0) return (size_t)g.C * g.H * g.W;         // the space-to-depth observation
    return t.implicit[gi] ? (size_t)0 : (size_t)g.Ho * g.Wo * g.ldc;
  };
  auto outp = [&](const ConvGeom& g, int Co) { return (size_t)g.Ho * g.Wo * Co; };
  f.clear(); u8.clear();
  switch (t.arch) {
    case DDRL_ARCH_ATARI: {
      // 0 cols1, 1 a1, 2 cols2, 3 a2, 4 cols3, 5 a3 | train: 6 da3, 7 dcols, 8 da2, 9 da1
      // fused first conv: tower 0 owns cols1 and the 2x-wide a1 / da1, tower 1 borrows them
      const size_t k0 = (t.fuse_role == 2 || (t.fuse_role == 1 && t.s2d_infer && (!train || t.s2d_train))) ? 0 : 1,
                   k1 = t.fuse_role == 2 ? 0 : (t.fuse_role == 1 ? 2 : 1);
      f = {k0 * cols(t.g[0]), k1 * outp(t.g[0], 32), cols(t.g[1]), outp(t.g[1], 64), cols(t.g[2]), outp(t.g[2], 64)};
      if (train) { f.push_back(outp(t.g[2], 64)); f.push_back(std::max(cols(t.g[1]), cols(t.g[2])));
                   f.push_back(outp(t.g[1], 64)); f.push_back(k1 * outp(t.g[0], 32)); }
      break;
    }
    case DDRL_ARCH_NAV:
    case DDRL_ARCH_NAVPED:
    case DDRL_ARCH_NAV1D: {
      const int C1 = 64, C2 = 128, C3 = 256;
      const ConvGeom *g0 = &t.g[0], *g1 = &t.g[1], *g2 = &t.g[2];
      const size_t p1 = (size_t)(g0->Ho / 2) * (g0->Wo / 2) * C1, p2 = (size_t)(g1->Ho / 2) * (g1->Wo / 2) * C2,
                   p3 = (size_t)(g2->Ho / 2) * (g2->Wo / 2) * C3;
      const int ldcat = t.arch == DDRL_ARCH_NAV1D ? 776 : 524;
      // 0 cols1, 1 z1, 2 p1, 3 cols2, 4 z2, 5 p2, 6 cols3, 7 z3, 8 p3, 9 cat, 10 f1
      const size_t own = t.borrow_cols ? 0 : 1;           // the observation-side im2col matrices are shared between unshared towers
      f = {own * cols(*g0), outp(*g0, C1), p1, cols(*g1), outp(*g1, C2), p2, cols(*g2), outp(*g2, C3), p3, (size_t)ldcat, 512};
      u8 = {p1, p2, p3};
      // 11 colsL1, 12 l1, 13 colsL2, 14 l2   (nav1d only; zero-sized otherwise)
      if (t.arch == DDRL_ARCH_NAV1D) { f.push_back(own * cols(t.g[3])); f.push_back(outp(t.g[3], 32));
                                       f.push_back(cols(t.g[4])); f.push_back(outp(t.g[4], 32)); }
      else { f.insert(f.end(), {0, 0, 0, 0}); }
      // 15 staging for NavPed channel concat (navped only)
      f.push_back(t.arch == DDRL_ARCH_NAVPED ? (size_t)t.in_ch * 48 * 48 : 0);
      if (train) {
        // 16 df1, 17 dcat, 18 dp3, 19 dz3, 20 dcols(max), 21 dp2, 22 dz2, 23 dp1, 24 dz1, 25 dl2, 26 dl1
        f.push_back(512); f.push_back(ldcat); f.push_back(p3); f.push_back(outp(*g2, C3));
        size_t dc = std::max(cols(*g1), cols(*g2));
        if (t.arch == DDRL_ARCH_NAV1D) dc = std::max(dc, cols(t.g[4]));
        f.push_back(dc); f.push_back(p2); f.push_back(outp(*g1, C2)); f.push_back(p1); f.push_back(outp(*g0, C1));
        if (t.arch == DDRL_ARCH_NAV1D) { f.push_back(outp(t.g[4], 32)); f.push_back(outp(t.g[3], 32)); }
        else { f.push_back(0); f.push_back(0); }
      }
      break;
    }
    case DDRL_ARCH_MLP:
      break;
  }
}

static size_t tower_bytes_per_sample(const Tower& t, bool train) {
  std::vector<size_t> f, u8;
  tower_sizes(t, train, f, u8);
  size_t b = 0;
  for (auto x : f) b += x * 4;
  for (auto x : u8) b += x;
  b += (size_t)t.feat * 4 * (train ? 2 : 1);
  return b;
}

static int ensure_workspace(ddrl_net* n, int B, bool train) {
  // micro-batch: bounded by a byte budget (DDRL_WS_GB, default 24 GiB) and DDRL_MICRO_BATCH (default 8192)
  size_t per = 0;
  for (auto& t : n->towers) per += tower_bytes_per_sample(t, train);
  per += (size_t)(n->ldA * 2 + 2 + 8) * 4;
  const size_t s2d_floats = (n->fuse_s2d && (!train || n->s2d_train)) ? (size_t)n->towers[0].g[0].C * n->towers[0].g[0].H * n->towers[0].g[0].W : 0;
  // (training workspaces only: one inference pass uses the observation once, and the extra pass over it costs more than the
  // first conv gains -- Forward 4.63 M vs 4.14 M actions/s, profiles/r4_notes.md; DDRL_PRESPLIT_INFER=1 forces it)
  const bool s2d_split = s2d_floats && tc3_mode(n) && s2d_floats % 8 == 0 && !getenv("DDRL_NO_PRESPLIT") &&
                         (train || getenv("DDRL_PRESPLIT_INFER"));
  per += s2d_floats * 4 * (s2d_split ? 2 : 1);
  const char* env_gb = getenv("DDRL_WS_GB");
  const char* env_mb = getenv("DDRL_MICRO_BATCH");
  const double budget = (env_gb ? atof(env_gb) : 24.0) * (double)(1ull << 30);
  int mb_cap = env_mb ? atoi(env_mb) : 8192;
  int mb = (int)std::min<double>((double)mb_cap, budget / (double)per);
  mb = std::max(mb, 1);
  if (mb >= 128) mb &= ~127;
  mb = std::min(mb, std::max(B, 1));
  if (n->ws.base && n->MB >= mb && (n->ws_train || !train)) return DDRL_OK;
  graphs_clear(n);                  // captured launches point into the old workspace
  for (const float* p : n->signbit_bases) tc3_signbits_unregister(p);
  n->signbit_bases.clear();
  if (n->ws.base) { cudaDeviceSynchronize(); cudaFree(n->ws.base); n->ws.base = nullptr; }
  // the amax registry is keyed by workspace pointers: start over (persistent entries are re-created on demand)
  for (auto it = n->amax_keys.begin(); it != n->amax_keys.end();) it = it->second.persistent ? std::next(it) : n->amax_keys.erase(it);
  for (auto& kv : n->amax_keys) kv.second.epoch = 0;
  n->amax_a_used = 0;
  n->MB = mb;
  n->ws_train = train;
  // total with per-buffer 256 B alignment slack
  size_t total = 0;
  for (auto& t : n->towers) {
    std::vector<size_t> f, u8;
    tower_sizes(t, train, f, u8);
    for (auto x : f) total += ((x * mb * 4 + 255) & ~size_t(255));
    for (auto x : u8) total += ((x * mb + 255) & ~size_t(255));
    total += 2 * (((size_t)t.feat * mb * 4 + 255) & ~size_t(255));
  }
  total += 4 * (((size_t)n->ldA * mb * 4 + 255) & ~size_t(255)) + 4096;
  total += 2 * (((size_t)kMaxExtra * mb * 4 + 255) & ~size_t(255));
  total += ((s2d_floats * mb * 4 + 255) & ~size_t(255)) * (s2d_split ? 2 : 1);
  // sign-bit tensors of the NatureCNN conv outputs (1 bit per element)
  const bool signbits = train && tc3_mode(n) && !getenv("DDRL_NO_SIGNBITS");
  if (signbits)
    for (auto& t : n->towers) {
      if (t.arch != DDRL_ARCH_ATARI) continue;
      std::vector<size_t> f, u8;
      tower_sizes(t, train, f, u8);
      for (int i : {1, 3, 5}) if (i < (int)f.size() && f[i]) total += ((f[i] * mb / 32 + 1) * 4 + 255) & ~size_t(255);
    }
  if (cudaMalloc(&n->ws.base, total) != cudaSuccess) {
    cudaGetLastError();
    n->ws.base = nullptr; n->MB = 0;
    return DDRL_E_NOMEM;
  }
  n->ws.cap = total; n->ws.used = 0;
  for (auto& t : n->towers) {
    std::vector<size_t> f, u8;
    tower_sizes(t, train, f, u8);
    t.buf.assign(f.size(), nullptr);
    t.idx.assign(u8.size(), nullptr);
    for (size_t i = 0; i < f.size(); ++i) if (f[i]) t.buf[i] = n->ws.take(f[i] * mb);
    for (size_t i = 0; i < u8.size(); ++i) t.idx[i] = reinterpret_cast<uint8_t*>(n->ws.take((u8[i] * mb + 3) / 4));
    t.h = n->ws.take((size_t)t.feat * mb);
    t.dh = train ? n->ws.take((size_t)t.feat * mb) : nullptr;
  }
  n->s2dbuf = s2d_floats ? n->ws.take(s2d_floats * mb) : nullptr;
  n->s2d16 = s2d_split ? n->ws.take(s2d_floats * mb) : nullptr;
  n->s2d16_plane = s2d_floats * mb * 2;
  if (signbits)
    for (auto& t : n->towers) {
      if (t.arch != DDRL_ARCH_ATARI) continue;
      std::vector<size_t> f, u8;
      tower_sizes(t, train, f, u8);
      for (int i : {1, 3, 5}) {
        if (i >= (int)f.size() || !f[i] || !t.buf[i] || (f[i] * mb) % 32 != 0) continue;     // (a borrowed a1 has f = 0: its owner registers it)
        float* w = n->ws.take(f[i] * mb / 32 + 1);
        if (!w) continue;
        tc3_signbits_register(t.buf[i], f[i] * mb, reinterpret_cast<unsigned int*>(w));
        n->signbit_bases.push_back(t.buf[i]);
      }
    }
  if (n->towers.size() == 2 && n->towers[1].borrow_cols) {
    Tower &t0 = n->towers[0], &t1 = n->towers[1];
    t1.buf[0] = t0.buf[0];
    if (t1.arch == DDRL_ARCH_NAV1D) t1.buf[11] = t0.buf[11];
  }
  if (n->fuse0) {
    Tower &t0 = n->towers[0], &t1 = n->towers[1];
    t1.buf[0] = t0.buf[0]; t1.buf[1] = t0.buf[1];
    if (train) t1.buf[9] = t0.buf[9];
  }
  n->logits = n->ws.take((size_t)n->ldA * mb);
  n->dlogits = n->ws.take((size_t)n->ldA * mb);
  n->vout = n->ws.take(mb);
  n->dv = n->ws.take(mb);
  n->vout_x = n->ws.take((size_t)kMaxExtra * mb);
  n->dv_x = n->ws.take((size_t)kMaxExtra * mb);
  return DDRL_OK;
}

// ---- packed weights -------------------------------------------------------------------
// packed layers in arena order; with the fused first conv the two towers' conv1 weights (and gradients) are adjacent, so
// [2 x Cout, K] is one GEMM operand
static std::vector<Lin*> packed_order(ddrl_net* n) {
  std::vector<Lin*> v;
  if (n->fuse0) { v.push_back(&n->towers[0].L[0]); v.push_back(&n->towers[1].L[0]); }
  for (auto& t : n->towers)
    for (size_t i = 0; i < t.L.size(); ++i)
      if (t.L[i].packed && !(n->fuse0 && i == 0)) v.push_back(&t.L[i]);
  return v;
}

static int alloc_packed(ddrl_net* n) {
  size_t bytes = 0;
  for (Lin* l : packed_order(n)) bytes += ((size_t)l->N * l->ldw * 4 + 255) & ~size_t(255);
  if (n->fuse0) {
    if (((size_t)n->towers[0].L[0].N * n->towers[0].L[0].ldw * 4) % 256 != 0) return DDRL_E_STATE;   // rows must abut
    DDRL_CUDA(cudaMalloc(&n->bias0c, sizeof(float) * 2 * n->towers[0].L[0].N));
  }
  const size_t w0s2d_off = bytes;                         // behind the layers' forward weights, inside the mirrored region
  if (n->fuse_s2d) bytes += ((size_t)2 * n->towers[0].L[0].N * n->towers[0].L[0].ldw * 4 + 255) & ~size_t(255);
  n->packed_grad_off = bytes;
  n->packed_grad_bytes = bytes;
  // data-gradient weights of the implicit convs (one re-packed copy per parity class), after the two twin regions
  size_t dg_bytes = 0;
  for (auto& t : n->towers)
    for (int i = 0; i < 5; ++i)
      for (auto& c : t.dg[i]) dg_bytes += ((size_t)t.g[i].C * c.K * 4 + 255) & ~size_t(255);
  for (auto& t : n->towers)
    for (int i = 0; i < 5; ++i)
      if (t.df[i].on) dg_bytes += ((size_t)t.df[i].N * t.df[i].K * 4 + 255) & ~size_t(255);
  n->packed_bytes = 2 * bytes + dg_bytes;
  if (!n->packed_bytes) return DDRL_OK;
  DDRL_CUDA(cudaMalloc(&n->packed_base, n->packed_bytes));
  DDRL_CUDA(cudaMemset(n->packed_base, 0, n->packed_bytes));     // padding columns stay zero forever
  if (tc2_mode(n)) {
    DDRL_CUDA(cudaMalloc(&n->split_base, 2 * n->packed_bytes));
    DDRL_CUDA(cudaMemset(n->split_base, 0, 2 * n->packed_bytes));
  }
  {
    size_t off = 2 * bytes;
    for (auto& t : n->towers)
      for (int i = 0; i < 5; ++i)
        for (auto& c : t.dg[i]) {
          c.wd = reinterpret_cast<float*>(n->packed_base + off);
          if (n->split_base) {
            c.wd_hi = reinterpret_cast<float*>(n->split_base + off);
            c.wd_lo = reinterpret_cast<float*>(n->split_base + n->packed_bytes + off);
          }
          off += ((size_t)t.g[i].C * c.K * 4 + 255) & ~size_t(255);
        }
    for (auto& t : n->towers)
      for (int i = 0; i < 5; ++i)
        if (t.df[i].on) {
          DgradFused& f = t.df[i];
          f.wd = reinterpret_cast<float*>(n->packed_base + off);
          f.wd_hi = reinterpret_cast<float*>(n->split_base + off);
          f.wd_lo = reinterpret_cast<float*>(n->split_base + n->packed_bytes + off);
          off += ((size_t)f.N * f.K * 4 + 255) & ~size_t(255);
        }
  }
  if (n->fuse_s2d) n->w0s2d = reinterpret_cast<float*>(n->packed_base + w0s2d_off);
  size_t off = 0;
  for (Lin* lp : packed_order(n)) {
    Lin& l = *lp;
    l.wp = reinterpret_cast<float*>(n->packed_base + off);
    l.dwp = reinterpret_cast<float*>(n->packed_base + n->packed_grad_off + off);
    if (n->split_base) {
      l.wp_hi = reinterpret_cast<float*>(n->split_base + off);
      l.wp_lo = reinterpret_cast<float*>(n->split_base + n->packed_bytes + off);
    }
    off += ((size_t)l.N * l.ldw * 4 + 255) & ~size_t(255);
  }
  if (tc3_mode(n)) {
    // every weight operand of a tcgen05 GEMM: layers (linear layers with their transposed twin for the data gradient),
    // data-gradient repacks of the implicit convs, the fused first conv's [2 Cout, K] operand and its s2d variant
    n->split_jobs.clear();
    auto add = [&](const float* w, int rows, int K, int ldw, W16* dst, bool tr) { n->split_jobs.push_back({w, rows, K, ldw, dst, tr}); };
    for (auto& t : n->towers)
      for (size_t i = 0; i < t.L.size(); ++i) {
        Lin& l = t.L[i];
        if (!l.packed || l.K < 32) continue;                      // thin first layers never reach the tensor-core engines
        if (n->fuse0 && i == 0) continue;                         // covered by the fused [2 Cout, K] operand
        const bool conv = i < 5 && t.conv_lin[i] == (int)i;
        add(l.wp, l.N, l.K, l.ldw, &l.w16, !conv);
      }
    if (n->fuse0) add(n->towers[0].L[0].wp, 2 * n->towers[0].L[0].N, n->towers[0].L[0].K, n->towers[0].L[0].ldw, &n->w16_fuse0, false);
    if (n->fuse_s2d) add(n->w0s2d, 2 * n->towers[0].L[0].N, n->towers[0].L[0].K, n->towers[0].L[0].ldw, &n->w16_s2d, false);
    for (auto& t : n->towers)
      for (int i = 0; i < 5; ++i) {
        for (auto& c : t.dg[i]) add(c.wd, t.g[i].C, c.K, c.K, &c.w16, false);
        if (t.df[i].on) add(t.df[i].wd, t.df[i].N, t.df[i].K, t.df[i].K, &t.df[i].w16, false);
      }
    if ((int)n->split_jobs.size() > kAmaxWeights / 2) return DDRL_E_UNSUPPORTED;
    size_t bytes16 = 0;
    auto r256 = [](size_t b) { return (b + 255) & ~size_t(255); };
    for (auto& j : n->split_jobs) {
      bytes16 += 2 * r256((size_t)j.rows * ((j.K + 7) & ~7) * 2);
      if (j.transposed) bytes16 += 2 * r256((size_t)j.K * ((j.rows + 7) & ~7) * 2);
    }
    n->h16_bytes = bytes16;
    DDRL_CUDA(cudaMalloc(&n->h16_base, bytes16));
    DDRL_CUDA(cudaMemset(n->h16_base, 0, bytes16));
    DDRL_CUDA(cudaMalloc(&n->amax_dev, sizeof(float) * kAmaxSlots));
    DDRL_CUDA(cudaMemset(n->amax_dev, 0, sizeof(float) * kAmaxSlots));
    size_t o16 = 0;
    n->w16_of.clear();
    for (auto& j : n->split_jobs) {
      W16& w = *j.dst;
      w.ld = (j.K + 7) & ~7;
      w.hi = n->h16_base + o16; o16 += r256((size_t)j.rows * w.ld * 2);
      w.lo = n->h16_base + o16; o16 += r256((size_t)j.rows * w.ld * 2);
      if (j.transposed) {
        w.ldT = (j.rows + 7) & ~7;
        w.hiT = n->h16_base + o16; o16 += r256((size_t)j.K * w.ldT * 2);
        w.loT = n->h16_base + o16; o16 += r256((size_t)j.K * w.ldT * 2);
      }
      w.amax = n->amax_dev + n->amax_w_used++;
      n->w16_of[j.w] = &w;
    }
  }
  return DDRL_OK;
}

static int side_init(ddrl_net* n) {
  if (n->ev_fork) return DDRL_OK;
  for (int k = 0; k < ddrl_net::kSide; ++k) {
    DDRL_CUDA(cudaStreamCreateWithFlags(&n->side[k], cudaStreamNonBlocking));
    DDRL_CUDA(cudaEventCreateWithFlags(&n->ev_join[k], cudaEventDisableTiming));
  }
  DDRL_CUDA(cudaEventCreateWithFlags(&n->ev_fork, cudaEventDisableTiming));
  return DDRL_OK;
}
static int side_fork(ddrl_net* n, cudaStream_t s) {
  DDRL_CUDA(cudaEventRecord(n->ev_fork, s));
  for (int k = 0; k < ddrl_net::kSide; ++k) DDRL_CUDA(cudaStreamWaitEvent(n->side[k], n->ev_fork, 0));
  return DDRL_OK;
}
static int side_join(ddrl_net* n, cudaStream_t s) {
  for (int k = 0; k < ddrl_net::kSide; ++k) {
    DDRL_CUDA(cudaEventRecord(n->ev_join[k], n->side[k]));
    DDRL_CUDA(cudaStreamWaitEvent(s, n->ev_join[k], 0));
  }
  return DDRL_OK;
}

// Emits the weight preparation.  phase_begin(k) is called before the launches of dependent phase k = 0, 1, 2 (the stream
// version joins / re-forks its side streams there; the recording version switches the job list).
template <class PhaseFn>
static int repack_emit(ddrl_net* n, cudaStream_t s0, bool par, PhaseFn&& phase_begin) {
  int rr = 0;
  cudaStream_t s = s0;
#define NEXT_STREAM() do { if (par) s = n->side[rr++ % ddrl_net::kSide]; } while (0)
  TRY(phase_begin(0));
  for (auto& t : n->towers)
    for (auto& l : t.L)
      if (l.packed) {
        NEXT_STREAM();
        if (l.s2d_s) TRY(pack_weight_s2d(n->params + n->T[l.w_t].offset, l.wp, l.N, l.s2d_C, l.s2d_KH, l.s2d_KW, l.s2d_s, l.ldw, s));
        else TRY(pack_weight(n->params + n->T[l.w_t].offset, l.wp, l.N, l.I, l.J, l.ldw, s));
      }
  for (auto& t : n->towers)
    for (int i = 0; i < 5; ++i)
      for (auto& c : t.dg[i]) {
        const Lin& l = t.L[t.conv_lin[i]];
        NEXT_STREAM();
        TRY(pack_dgrad(n->params + n->T[l.w_t].offset, t.g[i], l.N, c, s));
      }
  for (auto& t : n->towers)
    for (int i = 0; i < 5; ++i)
      if (t.df[i].on) {
        const Lin& l = t.L[t.conv_lin[i]];
        NEXT_STREAM();
        TRY(pack_dgrad_fused(n->params + n->T[l.w_t].offset, t.g[i], l.N, t.df[i], s));
      }
  if (n->fuse_s2d) {
    const ConvGeom& g = n->towers[0].g[0];
    for (int k = 0; k < 2; ++k) {
      const Lin& l = n->towers[k].L[0];
      NEXT_STREAM();
      TRY(pack_weight_s2d(n->params + n->T[l.w_t].offset, n->w0s2d + (size_t)k * l.N * l.ldw, l.N, g.C, g.KH, g.KW, g.stride, l.ldw, s));
    }
  }
  if (n->fuse0) {
    const Lin &l0 = n->towers[0].L[0], &l1 = n->towers[1].L[0];
    NEXT_STREAM();
    if (g_prep_rec) {
      PrepJob j{}; j.type = PREP_COPY; j.vblocks = 1;
      j.a = b_of(n, l0); j.b = n->bias0c; j.total = l0.N; prep_record(j);
      j.a = b_of(n, l1); j.b = n->bias0c + l0.N; j.total = l1.N; prep_record(j);
    } else {
      DDRL_CUDA(cudaMemcpyAsync(n->bias0c, b_of(n, l0), sizeof(float) * l0.N, cudaMemcpyDeviceToDevice, s));
      DDRL_CUDA(cudaMemcpyAsync(n->bias0c + l0.N, b_of(n, l1), sizeof(float) * l1.N, cudaMemcpyDeviceToDevice, s));
    }
  }
  if (g_prep_rec)                 // the stream version zeroes each amax slot right before its reduction (amax_f32)
    for (auto& j : n->split_jobs) {
      PrepJob z{}; z.type = PREP_ZERO; z.vblocks = 1; z.b = const_cast<float*>(j.dst->amax); z.total = 1; prep_record(z);
    }
  TRY(phase_begin(1));
  if (n->split_base) {
    NEXT_STREAM();
    // tf32 hi / lo mirrors of the forward weights [0, grad_off) and of the data-gradient weights [2*grad_off, end)
    const size_t fwd = n->packed_grad_off, dg0 = 2 * n->packed_grad_off, dgn = n->packed_bytes - dg0;
    char* hi = n->split_base;
    char* lo = n->split_base + n->packed_bytes;
    if (fwd) TRY(split_hi_lo(reinterpret_cast<float*>(n->packed_base), reinterpret_cast<float*>(hi), reinterpret_cast<float*>(lo),
                             (long long)(fwd / 4), s));
    if (dgn) TRY(split_hi_lo(reinterpret_cast<float*>(n->packed_base + dg0), reinterpret_cast<float*>(hi + dg0),
                             reinterpret_cast<float*>(lo + dg0), (long long)(dgn / 4), s));
  }
  if (g_prep_rec) {
    for (auto& j : n->split_jobs) TRY(amax_f32(j.w, j.rows, j.K, j.ldw, const_cast<float*>(j.dst->amax), true, s));
    TRY(phase_begin(2));
    for (auto& j : n->split_jobs) {
      W16& w = *j.dst;
      TRY(split_f16(j.w, j.rows, j.K, j.ldw, w.amax, const_cast<void*>(w.hi), const_cast<void*>(w.lo), w.ld, const_cast<void*>(w.hiT),
                    const_cast<void*>(w.loT), w.ldT, s));
    }
  } else {
    for (auto& j : n->split_jobs) {           // amax -> split of one operand stay on one stream
      W16& w = *j.dst;
      float* slot = const_cast<float*>(w.amax);
      NEXT_STREAM();
      TRY(amax_f32(j.w, j.rows, j.K, j.ldw, slot, true, s));
      TRY(split_f16(j.w, j.rows, j.K, j.ldw, slot, const_cast<void*>(w.hi), const_cast<void*>(w.lo), w.ld, const_cast<void*>(w.hiT),
                    const_cast<void*>(w.loT), w.ldT, s));
    }
    TRY(phase_begin(2));
  }
#undef NEXT_STREAM
  return DDRL_OK;
}

// gradient un-permutation (packed layout -> reference OIHW / [out, in]) of every packed layer (seg < 0), or of the layers
// whose gradient is final after backward segment `seg`
static int unpack_emit(ddrl_net* n, cudaStream_t s, int seg = -1) {
  if (n->s2d_train && (seg < 0 || seg == n->n_bwd_seg - 1)) {
    const ConvGeom& g = n->towers[0].g[0];
    const float* dw = reinterpret_cast<const float*>(reinterpret_cast<const char*>(n->w0s2d) + n->packed_grad_off);
    for (int k = 0; k < 2; ++k) {
      const Lin& l = n->towers[k].L[0];
      TRY(unpack_grad_s2d(dw + (size_t)k * l.N * l.ldw, n->grads + n->T[l.w_t].offset, l.N, g.C, g.KH, g.KW, g.stride, l.ldw, s));
    }
  }
  for (auto& t : n->towers)
    for (auto& l : t.L)
      if (l.packed) {
        if (n->s2d_train && &l == &t.L[0]) continue;         // done above from the fused space-to-depth gradient
        if (seg >= 0 && l.seg != seg) continue;
        if (l.s2d_s && !l.s2d_fwd_only) TRY(unpack_grad_s2d(l.dwp, n->grads + n->T[l.w_t].offset, l.N, l.s2d_C, l.s2d_KH, l.s2d_KW, l.s2d_s, l.ldw, s));
        else TRY(unpack_grad(l.dwp, n->grads + n->T[l.w_t].offset, l.N, l.I, l.J, l.ldw, s));
      }
  return DDRL_OK;
}

// Backward segments: tower t's backward is cut once, after the layers that hold most of its parameters (the linear stack on
// top of the conv stack); what runs before the cut of tower t belongs to segment t, the rest of the tower to segment t + 1, the
// cross-tower fused first conv (it runs after the last tower) to the last segment.  Segment k's gradients are final -- and
// un-permuted into the flat buffer -- when segment k ends.
static int tower_cut_layer(const Tower& t) {
  switch (t.arch) {
    case DDRL_ARCH_ATARI: return 3;                                  // fc 3136 -> 512 (6.4 of the tower's 6.7 MB)
    case DDRL_ARCH_NAV: case DDRL_ARCH_NAVPED: return 3;             // fc2, fc1, fc0 (flat -> 512: 18.9 MB) run first
    case DDRL_ARCH_NAV1D: return 6;
    default: return 0;
  }
}
static void assign_segments(ddrl_net* n) {
  const int T = (int)n->towers.size();
  n->n_bwd_seg = T + 1;
  for (int ti = 0; ti < T; ++ti) {
    Tower& t = n->towers[ti];
    const int cut = tower_cut_layer(t);
    for (int li = 0; li < (int)t.L.size(); ++li) {
      // ATARI / MLP run their layers top down (L.size()-1 .. 0); the nav towers run fc2, fc1, fc0 first (indices >= cut;
      // NAV1D: 8, 7, 6), then the conv stack and the laser branch
      t.L[li].seg = li >= cut ? ti : ti + 1;
      if (li == 0 && (t.fuse_role || n->s2d_train)) t.L[li].seg = T;
    }
  }
}

static bool prep_fused(const ddrl_net* n) {
  const char* e = getenv("DDRL_PREP_LAUNCHES");          // 1: one launch per layer and step (the round-1 behaviour)
  return !(e && e[0] == '1');
}

// builds the device job tables (synchronous allocations + copies: runs on the first preparation after bind, never inside a
// graph capture -- the first optimiser step and every `dirty` re-preparation go straight to the stream)
static int prep_build(ddrl_net* n) {
  PrepRecorder rec[3], unrec;
  assign_segments(n);
  std::vector<PrepRecorder> unrec_seg(n->n_bwd_seg);
  struct Guard { ~Guard() { g_prep_rec = nullptr; } } guard;
  int rc = repack_emit(n, nullptr, false, [&](int k) { g_prep_rec = &rec[k]; return DDRL_OK; });
  if (rc == DDRL_OK && n->grads) { g_prep_rec = &unrec; rc = unpack_emit(n, nullptr); }
  for (int k = 0; rc == DDRL_OK && n->grads && k < n->n_bwd_seg; ++k) { g_prep_rec = &unrec_seg[k]; rc = unpack_emit(n, nullptr, k); }
  g_prep_rec = nullptr;
  if (rc != DDRL_OK) return rc;
  for (int k = 0; k < 3; ++k) TRY(n->prep[k].upload(rec[k].jobs));
  TRY(n->unprep.upload(unrec.jobs));
  for (auto& t : n->unprep_seg) t.clear();
  n->unprep_seg.assign(n->n_bwd_seg, PrepTable());
  for (int k = 0; k < n->n_bwd_seg; ++k) TRY(n->unprep_seg[k].upload(unrec_seg[k].jobs));
  n->prep_ready = true;
  return DDRL_OK;
}

static int repack(ddrl_net* n, cudaStream_t s0) {
  if (prep_fused(n)) {
    if (!n->prep_ready) TRY(prep_build(n));
    TRY(n->prep[0].launch("prep_pack_kernel", s0));
    TRY(n->prep[1].launch("prep_amax_kernel", s0));
    TRY(n->prep[2].launch("prep_split_kernel", s0));
    n->dirty = false;
    return DDRL_OK;
  }
  // one launch per operand: fp32 re-packs on side streams; after a join, per weight operand amax -> fp16 split.  With the
  // profiler hooks on (per-launch events on ONE stream) everything stays on the caller's stream.
  const bool par = !g_prof_on && !getenv("DDRL_REPACK_SERIAL");
  if (par) TRY(side_init(n));
  TRY(repack_emit(n, s0, par, [&](int k) {
    if (!par) return DDRL_OK;
    if (k > 0) TRY(side_join(n, s0));
    if (k < 2) TRY(side_fork(n, s0));
    return DDRL_OK;
  }));
  n->dirty = false;
  return DDRL_OK;
}

// ---- CUDA-graph cache ------------------------------------------------------------------
static void graph_entry_destroy(ddrl_net::GraphEntry& e) {
  if (e.exec) cudaGraphExecDestroy(e.exec);
  if (e.graph) cudaGraphDestroy(e.graph);
  for (auto x : e.pre_execs) cudaGraphExecDestroy(x);
  for (auto g : e.pre_graphs) cudaGraphDestroy(g);
}
static void graphs_clear(ddrl_net* n) {
  for (auto& e : n->graphs) graph_entry_destroy(e);
  n->graphs.clear();
  n->mb_seen.clear();
}
// Segment cut of the backward pass (see ddrl_net::Capture): ends segment n->cap.seg.  Inside a capture the gradients of the
// segment are un-permuted, the current graph is closed and the next one opened; outside it does nothing.
static int seg_cut(ddrl_net* n, cudaStream_t s) {
  ddrl_net::Capture& c = n->cap;
  if (!c.active || c.failed || c.seg >= n->n_bwd_seg - 1 || (int)n->unprep_seg.size() != n->n_bwd_seg) return DDRL_OK;
  TRY(n->unprep_seg[c.seg].launch("prep_unpack_kernel", s));
  cudaGraph_t g = nullptr;
  if (cudaStreamEndCapture(s, &g) != cudaSuccess || !g) { c.failed = true; return DDRL_E_CUDA; }
  c.done.push_back(g);
  c.launches.push_back(g_launches - c.l0);
  c.l0 = g_launches;
  ++c.seg;
  if (cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal) != cudaSuccess) { c.failed = true; return DDRL_E_CUDA; }
  return DDRL_OK;
}
// the value clip needs the rollout's values of critic 0, and old values without a clip width would be ignored
static bool value_clip_ok(const ddrl_ppo_hparams* hp, const float* old_values) {
  return old_values ? hp->value_clip > 0.f : !(hp->value_clip > 0.f);
}
static bool graphs_enabled(ddrl_net* n) {
  const char* e = getenv("DDRL_NO_GRAPH");
  return !(e && e[0] == '1') && !n->graphs_off && !g_prof_on;
}
static std::string graph_key(const char* tag, std::initializer_list<const void*> ptrs, std::initializer_list<long long> ints,
                             const void* blob, size_t blob_bytes) {
  std::string k(tag);
  char b[40];
  for (const void* p : ptrs) { snprintf(b, sizeof(b), "|%p", p); k += b; }
  for (long long v : ints) { snprintf(b, sizeof(b), "|%lld", v); k += b; }
  k += '|';
  k.append(reinterpret_cast<const char*>(blob), blob_bytes);
  return k;
}
// Runs `body(stream)` through a cached graph: the first call with this key captures it on the net's private capture stream
// (nothing executes during capture; side-stream forks inside `body` become parallel branches), later calls replay.  A
// failed capture sets *off (default: n->graphs_off, all graphs of this net) and runs the body on the caller's stream.
template <class F>
static int run_graphed(ddrl_net* n, const std::string& key, cudaStream_t s, F&& body, ddrl_net::GraphEntry** out = nullptr,
                       bool* off = nullptr) {
  ddrl_net::GraphEntry* e = nullptr;
  for (auto& g : n->graphs) if (g.key == key) { e = &g; break; }
  if (!e) {
    if (!n->cap_stream) DDRL_CUDA(cudaStreamCreateWithFlags(&n->cap_stream, cudaStreamNonBlocking));
    TRY(side_init(n));
    const long long l0 = g_launches;
    ddrl_net::Capture& c = n->cap;
    c = ddrl_net::Capture();
    c.l0 = l0;
    DDRL_CUDA(cudaStreamBeginCapture(n->cap_stream, cudaStreamCaptureModeThreadLocal));
    c.active = true;
    const int rc = body(n->cap_stream);
    c.active = false;
    cudaGraph_t g = nullptr;
    const cudaError_t ce = cudaStreamEndCapture(n->cap_stream, &g);
    ddrl_net::GraphEntry ne;
    bool ok = rc == DDRL_OK && ce == cudaSuccess && g && !c.failed;
    for (size_t k = 0; ok && k < c.done.size(); ++k) {
      cudaGraphExec_t x = nullptr;
      ok = cudaGraphInstantiate(&x, c.done[k], 0) == cudaSuccess;
      if (ok) ne.pre_execs.push_back(x);
    }
    cudaGraphExec_t exec = nullptr;
    ok = ok && cudaGraphInstantiate(&exec, g, 0) == cudaSuccess;
    if (!ok) {
      if (g) cudaGraphDestroy(g);
      for (auto x : ne.pre_execs) cudaGraphExecDestroy(x);
      for (auto d : c.done) cudaGraphDestroy(d);
      c = ddrl_net::Capture();
      cudaGetLastError();
      g_launches = l0;
      *(off ? off : &n->graphs_off) = true;
      if (out) *out = nullptr;
      return body(s);
    }
    if (n->graphs.size() >= 8) {             // evict the least recently used entry
      size_t lru = 0;
      for (size_t i = 1; i < n->graphs.size(); ++i) if (n->graphs[i].used < n->graphs[lru].used) lru = i;
      graph_entry_destroy(n->graphs[lru]);
      n->graphs.erase(n->graphs.begin() + lru);
    }
    ne.key = key; ne.graph = g; ne.exec = exec;
    ne.pre_graphs = c.done;
    ne.pre_launches = c.launches;
    ne.launches = g_launches - c.l0;
    c = ddrl_net::Capture();
    g_launches = l0;
    n->graphs.push_back(ne);
    e = &n->graphs.back();
  }
  e->used = ++n->graph_clock;
  if (out) *out = e;
  else {
    for (size_t k = 0; k < e->pre_execs.size(); ++k) {
      DDRL_CUDA(cudaGraphLaunch(e->pre_execs[k], s));
      g_launches += e->pre_launches[k];
    }
    DDRL_CUDA(cudaGraphLaunch(e->exec, s));
    g_launches += e->launches;
  }
  return DDRL_OK;
}

// ---- encoder schedules ------------------------------------------------------------------
static int conv_block(const ddrl_net* n, const Tower& t, int gi, int li, const float* x, float* cols, float* y, int mb,
                      cudaStream_t s, bool cols_cached = false) {
  const bool s2d = gi == 0 && t.s2d0;
  if (s2d && !cols_cached) TRY(space_to_depth(t.g[0], x, cols, mb, s));
  const ConvGeom& g = s2d ? t.gs : t.g[gi];
  if (s2d || t.implicit[gi]) {
    const Lin& l = t.L[li];
    const bool sub = gi == 1 && t.in1_ctot;
    const ConvOp o = conv_op_fwd(g, s2d ? cols : x, sub ? t.in1_ctot : g.C, sub ? t.in1_coff : 0, mb);
    if (tc3_mode(n) && l.w16.hi) {
      ddrl_net* nn = const_cast<ddrl_net*>(n);
      const float* ama = nullptr;
      TRY(amax_in_slot(nn, o.a, (long long)mb * o.Hin * o.Win, o.Ctot, o.Ctot, s, &ama, s2d));
      return tc3_conv_fwd(o, l.w16.hi, l.w16.lo, l.w16.ld, l.N, ama, l.w16.amax, b_of(n, l), l.act, nullptr, y,
                          (long long)o.Yn * o.Xn * l.N, (long long)o.Xn * l.N, l.N,
                          amax_out_slot(nn, y, (long long)mb * o.Yn * o.Xn, l.N, l.N), s);
    }
    if (tc2_mode(n))
      return tc2_conv_fwd(o, l.wp_hi, l.wp_lo, l.ldw, l.N, b_of(n, l), l.act, nullptr, y, (long long)o.Yn * o.Xn * l.N,
                          (long long)o.Xn * l.N, l.N, s);
    return conv_tc_fwd(o, W_of(n, l), l.ldw, l.N, b_of(n, l), l.act, nullptr, y, (long long)o.Yn * o.Xn * l.N,
                       (long long)o.Xn * l.N, l.N, s);
  }
  if (!cols_cached) TRY(im2col(g, x, cols, mb, s));
  if (gi == 0) const_cast<ddrl_net*>(n)->amax_persist_next = true;     // observation-side im2col matrix
  return lin_fwd(n, t.L[li], cols, g.ldc, y, t.L[li].N, (long long)mb * g.Ho * g.Wo, s);
}

// reuse_obs: the im2col matrices of the layers that read the OBSERVATIONS are still valid from the previous call
// (PPO.learn runs TRAINING_ITER_TIME iterations over the same batch, nn/ppo.py:79-82)
static int tower_forward(ddrl_net* n, Tower& t, const float* const* obs, long long row0, int mb, bool train, cudaStream_t s,
                         bool reuse_obs = false) {
  auto& b = t.buf;
  switch (t.arch) {
    case DDRL_ARCH_ATARI: {
      const float* x = obs[0] + row0 * t.g[0].sb;
      if (!t.fuse_role) TRY(conv_block(n, t, 0, 0, x, b[0], b[1], mb, s, reuse_obs));     // else: fused_conv0_fwd ran it
      TRY(conv_block(n, t, 1, 1, b[1], b[2], b[3], mb, s));
      TRY(conv_block(n, t, 2, 2, b[3], b[4], b[5], mb, s));
      TRY(lin_fwd(n, t.L[3], b[5], 3136, t.h, 512, mb, s));
      return DDRL_OK;
    }
    case DDRL_ARCH_NAV:
    case DDRL_ARCH_NAVPED:
    case DDRL_ARCH_NAV1D: {
      const bool d1 = t.arch == DDRL_ARCH_NAV1D;
      const int ldcat = d1 ? 776 : 524;
      const float* img;
      if (t.arch == DDRL_ARCH_NAV) img = obs[0] + row0 * t.g[0].sb;
      else if (d1) img = obs[2] + row0 * t.g[0].sb;
      else {
        // NavPedPreNet: cat(state[0] [B,in_ch-3,48,48], state[2] [B,3,48,48]) along channels (nav_encoder.py:72)
        const int c0 = t.in_ch - 3, hw = 48 * 48;
        TRY(copy2d(obs[0] + row0 * c0 * hw, c0 * hw, b[15], t.in_ch * hw, mb, c0 * hw, s));
        TRY(copy2d(obs[2] + row0 * 3 * hw, 3 * hw, b[15] + c0 * hw, t.in_ch * hw, mb, 3 * hw, s));
        img = b[15];
      }
      const ConvGeom *g0 = &t.g[0], *g1 = &t.g[1], *g2 = &t.g[2];
      // tc3: the pooling kernels leave max|output| in the operand's amax slot (no reduction pass of its own per tensor)
      auto pool_slot = [&](const float* out, const ConvGeom* g, int C) {
        return amax_out_slot(const_cast<ddrl_net*>(n), out, (long long)mb * (g->Ho / 2) * (g->Wo / 2), C, C);
      };
      TRY(conv_block(n, t, 0, 0, img, b[0], b[1], mb, s, reuse_obs || t.borrow_cols));    // tower 0 ran first: its cols are current
      TRY(pool_fwd(b[1], b[2], t.idx[0], mb, g0->Ho, g0->Wo, 64, s, pool_slot(b[2], g0, 64)));
      TRY(conv_block(n, t, 1, 1, b[2], b[3], b[4], mb, s));
      TRY(pool_fwd(b[4], b[5], t.idx[1], mb, g1->Ho, g1->Wo, 128, s, pool_slot(b[5], g1, 128)));
      TRY(conv_block(n, t, 2, 2, b[5], b[6], b[7], mb, s));
      TRY(pool_fwd(b[7], b[8], t.idx[2], mb, g2->Ho, g2->Wo, 256, s, pool_slot(b[8], g2, 256)));
      const int flat = (g2->Ho / 2) * (g2->Wo / 2) * 256;
      const float* vec = obs[1];
      if (d1) {
        // laser branch: conv1d1 -> conv1d2 (no activation between, nav_encoder.py:109-110) -> fc_1d+relu -> cat[:, 0:256]
        const float* laser = obs[0] + row0 * t.g[3].sb;
        TRY(conv_block(n, t, 3, 3, laser, b[11], b[12], mb, s, reuse_obs || t.borrow_cols));
        TRY(conv_block(n, t, 4, 4, b[12], b[13], b[14], mb, s));
        TRY(lin_fwd(n, t.L[5], b[14], 7616, b[9], ldcat, mb, s));
        TRY(lin_fwd(n, t.L[6], b[8], flat, b[9] + 256, ldcat, mb, s));           // fc0 -> cat[:, 256:768]
        TRY(copy2d(vec + row0 * 5, 5, b[9] + 768, ldcat, mb, 5, s));             // vec -> cat[:, 768:773]
        TRY(lin_fwd(n, t.L[7], b[9], ldcat, b[10], 512, mb, s));
        TRY(lin_fwd(n, t.L[8], b[10], 512, t.h, 512, mb, s));
      } else {
        TRY(lin_fwd(n, t.L[3], b[8], flat, b[9], ldcat, mb, s));                 // fc0 -> cat[:, 0:512]
        TRY(copy2d(vec + row0 * 9, 9, b[9] + 512, ldcat, mb, 9, s));             // vec -> cat[:, 512:521]
        TRY(lin_fwd(n, t.L[4], b[9], ldcat, b[10], 512, mb, s));
        TRY(lin_fwd(n, t.L[5], b[10], 512, t.h, 512, mb, s));
      }
      return DDRL_OK;
    }
    case DDRL_ARCH_MLP:
      return lin_fwd(n, t.L[0], obs[0] + row0 * t.in_ch, t.in_ch, t.h, t.feat, mb, s);
  }
  return DDRL_E_ARG;
}

// conv layer backward.  dy [M, Cout] holds dL/d(pre-activation).  x: the layer's NHWC input (implicit path) / cols: its
// im2col matrix (explicit path).  db, dW, and -- if dx -- the input gradient times act'(x) (mask_act: activation that
// produced x; 0 = none or handled elsewhere, e.g. by pool_bwd)
static int conv_bwd(const ddrl_net* n, const Tower& t, int gi, int li, const float* x, const float* cols, float* dy,
                    float* dcols, float* dx, int mask_act, int mb, cudaStream_t s) {
  const bool s2d = gi == 0 && t.s2d0;
  const ConvGeom& g = s2d ? t.gs : t.g[gi];
  const Lin& l = t.L[li];
  const long long M = (long long)mb * g.Ho * g.Wo;
  if (s2d) {                                       // first layer: no data gradient; x2 = the cached space-to-depth tensor
    if (tc3_mode(n) && tc3_conv_wgrad_supported(conv_op_fwd(g, cols, g.C, 0, mb)) && !getenv("DDRL_TC3_NO_WGRAD")) {
      ddrl_net* nn = const_cast<ddrl_net*>(n);
      const float *amx = nullptr, *amy = nullptr;
      TRY(amax_in_slot(nn, cols, (long long)mb * g.H * g.W, g.C, g.C, s, &amx, true));
      TRY(amax_in_slot(nn, dy, M, l.N, l.N, s, &amy));
      if (!fuse_colsum()) TRY(colsum_add(dy, l.N, M, l.N, db_of(n, l), s));
      return tc3_conv_wgrad(conv_op_fwd(g, cols, g.C, 0, mb), dy, l.N, l.N, amx, amy, dW_of(n, l), l.ldw, s,
                            fuse_colsum() ? db_of(n, l) : nullptr);
    }
    TRY(colsum_add(dy, l.N, M, l.N, db_of(n, l), s));
    if (tc2_mode(n)) return tc2_conv_wgrad(conv_op_fwd(g, cols, g.C, 0, mb), dy, l.N, l.N, dW_of(n, l), l.ldw, s);
    return conv_tc_wgrad(conv_op_fwd(g, cols, g.C, 0, mb), dy, l.N, l.N, dW_of(n, l), l.ldw, s);
  }
  if (t.implicit[gi]) {
    const bool sub = gi == 1 && t.in1_ctot;
    const int ctot = sub ? t.in1_ctot : g.C, coff = sub ? t.in1_coff : 0;
    const bool w3 = tc3_mode(n) && tc3_conv_wgrad_supported(conv_op_fwd(g, x, ctot, coff, mb)) && !getenv("DDRL_TC3_NO_WGRAD");
    if (!(w3 && fuse_colsum())) TRY(colsum_add(dy, l.N, M, l.N, db_of(n, l), s));
    if (w3) {
      ddrl_net* nn = const_cast<ddrl_net*>(n);
      const float *amx = nullptr, *amy = nullptr;
      TRY(amax_in_slot(nn, x, (long long)mb * g.H * g.W, ctot, ctot, s, &amx));
      TRY(amax_in_slot(nn, dy, M, l.N, l.N, s, &amy));
      TRY(tc3_conv_wgrad(conv_op_fwd(g, x, ctot, coff, mb), dy, l.N, l.N, amx, amy, dW_of(n, l), l.ldw, s,
                         fuse_colsum() ? db_of(n, l) : nullptr));
    } else {
      if (tc2_mode(n)) TRY(tc2_conv_wgrad(conv_op_fwd(g, x, ctot, coff, mb), dy, l.N, l.N, dW_of(n, l), l.ldw, s));
      else TRY(conv_tc_wgrad(conv_op_fwd(g, x, ctot, coff, mb), dy, l.N, l.N, dW_of(n, l), l.ldw, s));
    }
    Tc3Ctx ctx{nullptr, nullptr};
    const bool t3 = tc3_mode(n) && dx && (t.df[gi].on ? t.df[gi].w16.hi != nullptr : (!t.dg[gi].empty() && t.dg[gi][0].w16.hi != nullptr));
    if (t3) {
      ddrl_net* nn = const_cast<ddrl_net*>(n);
      TRY(amax_in_slot(nn, dy, M, l.N, l.N, s, &ctx.amax_a));
      // a data gradient that fills a channel slice of a wider tensor (the towers' halves of the fused first conv's output
      // gradient) accumulates into the slot of the WHOLE tensor: every slice is written in this pass by a tracked producer,
      // so after the last of them the slot holds the tensor's amax (atomicMax; zeroed at the start of the pass)
      ctx.amax_out = amax_out_slot(nn, dx, (long long)mb * g.H * g.W, sub ? ctot : g.C, sub ? ctot : g.C);
    }
    if (dx && t.df[gi].on)
      TRY(conv_dgrad_fused_tc2(g, l.N, t.df[gi], dy, dx, mask_act ? mask_act + 2 : 0, mask_act ? x : nullptr, mb, s, ctot, coff,
                               t3 ? &ctx : nullptr));
    else if (dx && sub) return DDRL_E_STATE;
    else if (dx)
      TRY(conv_dgrad_tc(g, l.N, t.dg[gi], dy, l.N, 0, dx, mask_act ? mask_act + 2 : 0, mask_act ? x : nullptr, mb, s,
                        tc2_mode(n), t3 ? &ctx : nullptr));
    return DDRL_OK;
  }
  if (gi == 0) const_cast<ddrl_net*>(n)->amax_persist_next = true;     // observation-side im2col matrix
  TRY(lin_bwd(n, l, cols, g.ldc, dy, l.N, dx ? dcols : nullptr, g.ldc, g.ldc, 0, nullptr, M, s));
  if (dx) {
    TRY(col2im(g, dcols, dx, mb, s));
    if (mask_act) TRY(act_bwd(dx, g.C, x, g.C, (long long)mb * g.H * g.W, g.C, mask_act, s));
  }
  return DDRL_OK;
}

static int tower_backward(ddrl_net* n, Tower& t, const float* const* obs, long long row0, int mb, cudaStream_t s) {
  auto& b = t.buf;
  switch (t.arch) {
    case DDRL_ARCH_ATARI: {
      // t.dh = dL/dh (linear has no activation); every conv output went through leaky_relu (atari_encoder.py:26-28)
      TRY(lin_bwd(n, t.L[3], b[5], 3136, t.dh, 512, b[6], 3136, 3136, ACT_LEAKY, b[5], mb, s));
      TRY(seg_cut(n, s));
      TRY(conv_bwd(n, t, 2, 2, b[3], b[4], b[6], b[7], b[8], ACT_LEAKY, mb, s));
      TRY(conv_bwd(n, t, 1, 1, b[1], b[2], b[8], b[7], b[9], ACT_LEAKY, mb, s));
      if (!t.fuse_role) TRY(conv_bwd(n, t, 0, 0, nullptr, b[0], b[9], nullptr, nullptr, 0, mb, s));   // else: fused_conv0_bwd
      return DDRL_OK;
    }
    case DDRL_ARCH_NAV:
    case DDRL_ARCH_NAVPED:
    case DDRL_ARCH_NAV1D: {
      const bool d1 = t.arch == DDRL_ARCH_NAV1D;
      const int ldcat = d1 ? 776 : 524;
      const ConvGeom *g0 = &t.g[0], *g1 = &t.g[1], *g2 = &t.g[2];
      const int flat = (g2->Ho / 2) * (g2->Wo / 2) * 256;
      float *df1 = b[16], *dcat = b[17], *dp3 = b[18], *dz3 = b[19], *dcols = b[20], *dp2 = b[21], *dz2 = b[22],
            *dp1 = b[23], *dz1 = b[24];
      const int Lfc2 = d1 ? 8 : 5, Lfc1 = d1 ? 7 : 4, Lfc0 = d1 ? 6 : 3;
      const int img_off = d1 ? 256 : 0;
      auto unpool_slot = [&](const float* da, const ConvGeom* g, int C) {
        return amax_out_slot(n, da, (long long)mb * g->Ho * g->Wo, C, C);
      };
      // fc2 (no activation) <- relu(fc1) <- relu(cat parts): each data gradient is multiplied by relu' of its target
      TRY(lin_bwd(n, t.L[Lfc2], b[10], 512, t.dh, 512, df1, 512, 512, ACT_RELU, b[10], mb, s));
      TRY(lin_bwd(n, t.L[Lfc1], b[9], ldcat, df1, 512, dcat, ldcat, img_off + 512, ACT_RELU, b[9], mb, s));
      TRY(lin_bwd(n, t.L[Lfc0], b[8], flat, dcat + img_off, ldcat, dp3, flat, flat, 0, nullptr, mb, s));
      TRY(seg_cut(n, s));
      // ReLU' of the conv outputs is folded into pool_bwd (a > 0 test)
      TRY(pool_bwd(dp3, t.idx[2], b[7], dz3, mb, g2->Ho, g2->Wo, 256, s, unpool_slot(dz3, g2, 256)));
      TRY(conv_bwd(n, t, 2, 2, b[5], b[6], dz3, dcols, dp2, 0, mb, s));
      TRY(pool_bwd(dp2, t.idx[1], b[4], dz2, mb, g1->Ho, g1->Wo, 128, s, unpool_slot(dz2, g1, 128)));
      TRY(conv_bwd(n, t, 1, 1, b[2], b[3], dz2, dcols, dp1, 0, mb, s));
      TRY(pool_bwd(dp1, t.idx[0], b[1], dz1, mb, g0->Ho, g0->Wo, 64, s, unpool_slot(dz1, g0, 64)));
      TRY(conv_bwd(n, t, 0, 0, nullptr, b[0], dz1, nullptr, nullptr, 0, mb, s));
      if (d1) {
        // laser branch: fc_1d+relu <- conv1d2 <- conv1d1, no activation between the convs (nav_encoder.py:109-110)
        float *dl2 = b[25], *dl1 = b[26];
        TRY(lin_bwd(n, t.L[5], b[14], 7616, dcat, ldcat, dl2, 7616, 7616, 0, nullptr, mb, s));
        TRY(conv_bwd(n, t, 4, 4, b[12], b[13], dl2, dcols, dl1, 0, mb, s));
        TRY(conv_bwd(n, t, 3, 3, nullptr, b[11], dl1, nullptr, nullptr, 0, mb, s));
      }
      return DDRL_OK;
    }
    case DDRL_ARCH_MLP: {
      TRY(act_bwd(t.dh, t.feat, t.h, t.feat, mb, t.feat, ACT_RELU, s));
      TRY(lin_bwd(n, t.L[0], obs[0] + row0 * t.in_ch, t.in_ch, t.dh, t.feat, nullptr, 0, 0, 0, nullptr, mb, s));
      return seg_cut(n, s);
    }
  }
  return DDRL_E_ARG;
}

static int check_obs(const ddrl_net* n, const float* const* obs, int n_obs) {
  const int need = ddrl_net_num_obs(n);
  if (!obs || n_obs < need) return DDRL_E_ARG;
  for (int i = 0; i < need; ++i)
    if (!obs[i] && ddrl_net_obs_elems(n, i) > 0) return DDRL_E_ARG;
  return DDRL_OK;
}

// First conv of both unshared towers in one pass over the shared im2col matrix: a1c[M, 2 Cout] = act(cols W01^T + b01)
// (rows 0..Cout-1 of W01 = actor tower, the rest = critic tower; each tower's conv2 reads its channel half).
static int fused_conv0_fwd(ddrl_net* n, const float* const* obs, long long row0, int mb, bool train, cudaStream_t s,
                           bool cols_cached) {
  Tower& t0 = n->towers[0];
  const ConvGeom& g = t0.g[0];
  const Lin& l = t0.L[0];
  if (n->fuse_s2d && (n->s2d_train || (!train && !n->ws_train))) {
    const ConvGeom& gs = t0.gs;
    const ConvOp o = conv_op_fwd(gs, n->s2dbuf, gs.C, 0, mb);
    if (!cols_cached) {
      // tc3: the staging kernel leaves the operand's amax in its (persistent) slot on the way -- no reduction pass of its own
      float* slot = nullptr;
      if (tc3_mode(n) && n->w16_s2d.hi && n->amax_dev) {
        const std::string key = amax_key(n->s2dbuf, (long long)mb * o.Hin * o.Win, o.Ctot, o.Ctot);
        const int si = amax_slot_index(n, key, true);
        if (si >= 0) {
          slot = n->amax_dev + si;
          DDRL_CUDA(cudaMemsetAsync(slot, 0, sizeof(float), s));
          n->amax_keys[key].epoch = n->amax_epoch;
        }
      }
      TRY(space_to_depth(g, obs[0] + row0 * g.sb, n->s2dbuf, mb, s, slot));
    }
    const int N2 = 2 * l.N;
    if (tc3_mode(n) && n->w16_s2d.hi) {
      const float* ama = nullptr;
      TRY(amax_in_slot(n, n->s2dbuf, (long long)mb * o.Hin * o.Win, o.Ctot, o.Ctot, s, &ama, true));
      const void *p_hi = nullptr, *p_lo = nullptr;
      if (n->s2d16 && o.Cin % 64 == 0 && (train || getenv("DDRL_PRESPLIT_INFER"))) {
        p_hi = n->s2d16; p_lo = reinterpret_cast<const char*>(n->s2d16) + n->s2d16_plane;
        if (!cols_cached)
          TRY(tc3_presplit(n->s2dbuf, (long long)mb * o.Hin * o.Win * o.Ctot, ama, n->s2d16, reinterpret_cast<char*>(n->s2d16) + n->s2d16_plane, s));
      }
      return tc3_conv_fwd(o, n->w16_s2d.hi, n->w16_s2d.lo, n->w16_s2d.ld, N2, ama, n->w16_s2d.amax, n->bias0c, l.act, nullptr, t0.buf[1],
                          (long long)o.Yn * o.Xn * N2, (long long)o.Xn * N2, N2,
                          amax_out_slot(n, t0.buf[1], (long long)mb * o.Yn * o.Xn, N2, N2), s, nullptr, p_hi, p_lo);
    }
    return tc2_conv_fwd(o, hi_of(n, n->w0s2d), lo_of(n, n->w0s2d), l.ldw, N2, n->bias0c, l.act, nullptr, t0.buf[1], (long long)o.Yn * o.Xn * N2,
                        (long long)o.Xn * N2, N2, s);
  }
  if (!cols_cached) TRY(im2col(g, obs[0] + row0 * g.sb, t0.buf[0], mb, s));
  n->amax_persist_next = true;                       // the im2col matrix of the observations survives the learn call's iterations
  return gemm(n, 0, (int)((long long)mb * g.Ho * g.Wo), 2 * l.N, l.K, t0.buf[0], g.ldc, l.wp, l.ldw, t0.buf[1], 2 * l.N, n->bias0c,
              l.act, 0, 0, s);
}
// ... and its backward: da1c [M, 2 Cout] holds both towers' dL/d(pre-activation) side by side
static int fused_conv0_bwd(ddrl_net* n, int mb, cudaStream_t s) {
  Tower &t0 = n->towers[0], &t1 = n->towers[1];
  const ConvGeom& g = t0.g[0];
  const Lin &l0 = t0.L[0], &l1 = t1.L[0];
  const long long M = (long long)mb * g.Ho * g.Wo;
  float* dy = t0.buf[9];
  const bool w3 = tc3_mode(n) && !getenv("DDRL_TC3_NO_WGRAD");
  const bool fcs = fuse_colsum() && (n->s2d_train || w3);
  if (!fcs) TRY(colsum_add(dy, 2 * l0.N, M, l0.N + l1.N, db_of(n, l0), s, db_of(n, l1), l0.N));     // ONE pass over the fused gradient
  if (n->s2d_train) {
    // weight gradient of both towers in the space-to-depth K order: dW0s2d [2 Cout, K] (the twin of w0s2d in the gradient
    // half of the packed arena), un-permuted per tower after the micro-batch loop
    const ConvOp o = conv_op_fwd(t0.gs, n->s2dbuf, t0.gs.C, 0, mb);
    const float *amx = nullptr, *amy = nullptr;
    TRY(amax_in_slot(n, n->s2dbuf, (long long)mb * o.Hin * o.Win, o.Ctot, o.Ctot, s, &amx, true));
    TRY(amax_in_slot(n, dy, M, 2 * l0.N, 2 * l0.N, s, &amy));
    float* dw = reinterpret_cast<float*>(reinterpret_cast<char*>(n->w0s2d) + n->packed_grad_off);
    const bool psw = n->s2d16 && o.Cin % 64 == 0 && !getenv("DDRL_NO_PRESPLIT_WGRAD");
    return tc3_conv_wgrad(o, dy, 2 * l0.N, 2 * l0.N, amx, amy, dw, l0.ldw, s, fcs ? db_of(n, l0) : nullptr, fcs ? db_of(n, l1) : nullptr,
                          l0.N, psw ? n->s2d16 : nullptr, psw ? reinterpret_cast<const char*>(n->s2d16) + n->s2d16_plane : nullptr);
  }
  if (w3) {
    const float *amx = nullptr, *amy = nullptr;
    TRY(amax_in_slot(n, t0.buf[0], M, l0.K, g.ldc, s, &amx, true));
    TRY(amax_in_slot(n, dy, M, 2 * l0.N, 2 * l0.N, s, &amy));
    return tc3_wgrad(l0.K, 2 * l0.N, M, t0.buf[0], g.ldc, dy, 2 * l0.N, amx, amy, l0.dwp, l0.ldw, s, fcs ? db_of(n, l0) : nullptr,
                     fcs ? db_of(n, l1) : nullptr, l0.N);
  }
  return tc2_wgrad(l0.K, 2 * l0.N, M, t0.buf[0], g.ldc, dy, 2 * l0.N, l0.dwp, l0.ldw, s);
}

// encoders + heads for rows [row0, row0+mb): fills n->logits [mb, ldA], n->vout [mb]
static int forward_chunk(ddrl_net* n, const float* const* obs, long long row0, int mb, bool train, cudaStream_t s,
                         bool reuse_obs = false) {
  if (n->fuse0) TRY(fused_conv0_fwd(n, obs, row0, mb, train, s, reuse_obs));
  for (auto& t : n->towers) TRY(tower_forward(n, t, obs, row0, mb, train, s, reuse_obs));
  Tower& ta = n->towers[0];
  Tower& tc = n->towers[n->d.shared ? 0 : 1];
  const int A = n->d.act_dim, F = n->d.feat;
  TRY(skinny_fwd(ta.h, F, n->params + n->T[n->t_aw].offset, n->params + n->T[n->t_ab].offset, mb, A, F, n->logits, n->ldA, s));
  TRY(skinny_fwd(tc.h, F, n->params + n->T[n->t_cw].offset, n->params + n->T[n->t_cb].offset, mb, 1, F, n->vout, 1, s));
  for (size_t k = 0; k < n->extra.size(); ++k)       // [critic(states) for critic in self._critics], nn/ppo.py:75
    TRY(skinny_fwd(tc.h, F, n->extra[k].w, n->extra[k].b, mb, 1, F, n->vout_x + k * (size_t)n->MB, 1, s));
  return DDRL_OK;
}

}  // namespace ddrl

// =========================================================================================
// C ABI
// =========================================================================================
extern "C" int ddrl_net_create(const ddrl_net_desc* desc, ddrl_net** out) {
  if (!desc || !out) return DDRL_E_ARG;
  if (desc->arch < 0 || desc->arch > DDRL_ARCH_MLP || desc->act_dim < 1 || desc->in_ch < 1) return DDRL_E_ARG;
  if (desc->dist == DDRL_DIST_CATEGORICAL && desc->act_dim > 64) return DDRL_E_UNSUPPORTED;
  if (desc->dist == DDRL_DIST_GAUSSIAN && desc->act_dim > 8) return DDRL_E_UNSUPPORTED;
  if (desc->arch == DDRL_ARCH_NAVPED && desc->in_ch < 4) return DDRL_E_ARG;
  ddrl_net* n = new ddrl_net();
  n->d = *desc;
  if (n->d.arch != DDRL_ARCH_MLP) n->d.feat = 512;
  if (n->d.feat < 1) { delete n; return DDRL_E_ARG; }
  const int F = n->d.feat;
  // ---- parameter table: reference named_parameters() order (nn/ppo.py:26-30, actor.py:12-16,52-56, critic.py:8-12)
  if (n->d.shared) add_encoder_tensors(n, "prenet.", n->d.arch, n->d.in_ch, F);
  if (n->d.dist == DDRL_DIST_GAUSSIAN) add_tensor(n, "actor.log_std", {n->d.act_dim});
  if (!n->d.shared) add_encoder_tensors(n, "actor.pre.", n->d.arch, n->d.in_ch, F);
  add_tensor(n, "actor.actor_linear.weight", {n->d.act_dim, F});
  add_tensor(n, "actor.actor_linear.bias", {n->d.act_dim});
  const int64_t critic_begin = n->P;
  add_tensor(n, "critic.critic_linear.weight", {1, F});
  add_tensor(n, "critic.critic_linear.bias", {1});
  if (!n->d.shared) add_encoder_tensors(n, "critic.pre.", n->d.arch, n->d.in_ch, F);
  n->t_aw = find_tensor(n, "actor.actor_linear.weight");
  n->t_ab = find_tensor(n, "actor.actor_linear.bias");
  n->t_cw = find_tensor(n, "critic.critic_linear.weight");
  n->t_cb = find_tensor(n, "critic.critic_linear.bias");
  n->t_logstd = find_tensor(n, "actor.log_std");
  n->ldA = round4(n->d.act_dim);
  // Adam segments: shared -> one optimiser over everything (ppo.py:40); unshared -> actor_optim over
  // actor.* and critic_optim over critic.* (ppo.py:41-42), contiguous in the flat order
  if (n->d.shared) { n->nseg = 1; n->seg_begin[0] = 0; n->seg_begin[1] = n->P; }
  else { n->nseg = 2; n->seg_begin[0] = 0; n->seg_begin[1] = critic_begin; n->seg_begin[2] = n->P; }
  if (n->d.shared) {
    n->towers.resize(1);
    build_tower(n, n->towers[0], "prenet.", n->d.arch, n->d.in_ch, F);
  } else {
    n->towers.resize(2);
    build_tower(n, n->towers[0], "actor.pre.", n->d.arch, n->d.in_ch, F);
    build_tower(n, n->towers[1], "critic.pre.", n->d.arch, n->d.in_ch, F);
    // unshared towers read the same observation: run their first (explicit-im2col) conv as one N = 2 x Cout GEMM
    Tower &t0 = n->towers[0], &t1 = n->towers[1];
    {
      const char* nb = getenv("DDRL_NO_SHARED_COLS");
      const bool nav = n->d.arch == DDRL_ARCH_NAV1D || n->d.arch == DDRL_ARCH_NAV;
      if (nav && !(nb && nb[0] == '1') && !t0.implicit[0] && !t1.implicit[0] && !t0.s2d0) t1.borrow_cols = true;
    }
    const char* nf = getenv("DDRL_NO_FUSE0");
    if (n->d.arch == DDRL_ARCH_ATARI && tc2_mode(n) && !(nf && nf[0] == '1') && !t0.s2d0 && !t0.implicit[0] && t0.implicit[1] &&
        t0.df[1].on && t1.df[1].on && t0.L[0].N % 32 == 0 && 2 * t0.L[0].N <= 128 && t0.g[0].ldc % 4 == 0) {
      n->fuse0 = true;
      t0.fuse_role = 1; t1.fuse_role = 2;
      t0.in1_ctot = t1.in1_ctot = 2 * t0.L[0].N;
      t0.in1_coff = 0; t1.in1_coff = t0.L[0].N;
      const ConvGeom& g = t0.g[0];
      const int st = g.stride;
      const char* ns = getenv("DDRL_NO_S2D_FWD");
      if (!(ns && ns[0] == '1') && g.order == 1 && g.sw == 1 && g.pad == 0 && st > 1 && g.KH % st == 0 && g.KW % st == 0 &&
          g.H % st == 0 && g.W % st == 0 && (st * st * g.C) % 32 == 0 && (size_t)g.C * st * g.W * 4 <= 48 * 1024) {
        ConvGeom gs = conv_geom(g.H / st, g.W / st, st * st * g.C, false, g.KH / st, g.KW / st, 1, 0);
        static const float* const kAligned = reinterpret_cast<const float*>(uintptr_t(256));
        if (gs.Ho == g.Ho && gs.Wo == g.Wo && gs.K == g.K && conv_tc_supported(conv_op_fwd(gs, kAligned, gs.C, 0, 1), false)) {
          n->fuse_s2d = true;
          t0.gs = gs;
          t0.s2d_infer = true;
          const char* nst = getenv("DDRL_NO_S2D_TRAIN");
          if (tc3_mode(n) && !(nst && nst[0] == '1') && tc3_conv_wgrad_supported(conv_op_fwd(gs, kAligned, gs.C, 0, 1))) {
            n->s2d_train = true;
            t0.s2d_train = true;
          }
        }
      }
    }
  }
  *out = n;
  return DDRL_OK;
}

extern "C" int ddrl_net_destroy(ddrl_net* n) {
  if (!n) return DDRL_OK;
  graphs_clear(n);
  for (int k = 0; k < 3; ++k) n->prep[k].clear();
  n->unprep.clear();
  for (auto& t : n->unprep_seg) t.clear();
  if (n->cap_stream) cudaStreamDestroy(n->cap_stream);
  if (n->sumsq_dev) cudaFree(n->sumsq_dev);
  for (const float* p : n->signbit_bases) tc3_signbits_unregister(p);
  if (n->ws.base) cudaFree(n->ws.base);
  if (n->packed_base) cudaFree(n->packed_base);
  if (n->split_base) cudaFree(n->split_base);
  if (n->ev_fork) {
    for (int k = 0; k < ddrl_net::kSide; ++k) { cudaStreamDestroy(n->side[k]); cudaEventDestroy(n->ev_join[k]); }
    cudaEventDestroy(n->ev_fork);
  }
  if (n->h16_base) cudaFree(n->h16_base);
  if (n->amax_dev) cudaFree(n->amax_dev);
  if (n->bias0c) cudaFree(n->bias0c);
  delete n;
  return DDRL_OK;
}

extern "C" int ddrl_net_num_tensors(const ddrl_net* n) { return n ? (int)n->T.size() : DDRL_E_ARG; }
extern "C" int64_t ddrl_net_num_params(const ddrl_net* n) { return n ? n->P : DDRL_E_ARG; }
extern "C" int ddrl_net_tensor_info(const ddrl_net* n, int i, char* name, int name_cap, int64_t* shape4, int* ndim,
                                    int64_t* offset) {
  if (!n || i < 0 || i >= (int)n->T.size()) return DDRL_E_ARG;
  const TensorInfo& t = n->T[i];
  if (name && name_cap > 0) { strncpy(name, t.name.c_str(), name_cap - 1); name[name_cap - 1] = 0; }
  if (shape4) for (int k = 0; k < 4; ++k) shape4[k] = t.shape[k];
  if (ndim) *ndim = t.ndim;
  if (offset) *offset = t.offset;
  return DDRL_OK;
}

extern "C" int ddrl_net_bind(ddrl_net* n, float* params, float* grads, float* adam_m, float* adam_v) {
  if (!n || !params) return DDRL_E_ARG;
  n->params = params; n->grads = grads; n->am = adam_m; n->av = adam_v;
  n->dirty = true;
  graphs_clear(n);
  n->prep_ready = false;
  if (!n->packed_base) TRY(alloc_packed(n));
  return DDRL_OK;
}

extern "C" int ddrl_net_set_extra_critics(ddrl_net* n, int count, const float* const* w, const float* const* b,
                                          float* const* dw, float* const* db, const int* in_loss) {
  if (!n || count < 0 || count > kMaxExtra) return DDRL_E_ARG;
  if (count > 0 && !n->d.shared) return DDRL_E_UNSUPPORTED;     // an unshared extra critic owns an encoder: a net of its own
  if (count > 0 && (!w || !b)) return DDRL_E_ARG;
  n->extra.clear();
  graphs_clear(n);
  for (int k = 0; k < count; ++k) {
    if (!w[k] || !b[k]) return DDRL_E_ARG;
    const int on = in_loss ? in_loss[k] : 0;
    if (on && (!dw || !db || !dw[k] || !db[k])) return DDRL_E_ARG;
    n->extra.push_back({w[k], b[k], dw ? dw[k] : nullptr, db ? db[k] : nullptr, on});
  }
  return DDRL_OK;
}

extern "C" int ddrl_net_params_changed(ddrl_net* n) {
  if (!n) return DDRL_E_ARG;
  n->dirty = true;
  return DDRL_OK;
}

extern "C" int ddrl_net_num_obs(const ddrl_net* n) {
  if (!n) return DDRL_E_ARG;
  switch (n->d.arch) {
    case DDRL_ARCH_ATARI: case DDRL_ARCH_MLP: return 1;
    case DDRL_ARCH_NAV: return 2;
    default: return 3;
  }
}
extern "C" int64_t ddrl_net_obs_elems(const ddrl_net* n, int slot) {
  if (!n) return DDRL_E_ARG;
  switch (n->d.arch) {
    case DDRL_ARCH_ATARI: return slot == 0 ? (int64_t)n->d.in_ch * 84 * 84 : 0;
    case DDRL_ARCH_MLP: return slot == 0 ? n->d.in_ch : 0;
    case DDRL_ARCH_NAV: return slot == 0 ? (int64_t)n->d.in_ch * 48 * 48 : (slot == 1 ? 9 : 0);
    case DDRL_ARCH_NAVPED: return slot == 0 ? (int64_t)(n->d.in_ch - 3) * 48 * 48 : (slot == 1 ? 9 : (slot == 2 ? 3 * 48 * 48 : 0));
    case DDRL_ARCH_NAV1D: return slot == 0 ? 960 * (int64_t)laser_ch_of(n) : (slot == 1 ? 5 : (slot == 2 ? (int64_t)n->d.in_ch * 48 * 48 : 0));
  }
  return 0;
}
extern "C" int64_t ddrl_net_workspace_bytes(const ddrl_net* n) { return n ? (int64_t)(n->ws.cap + n->packed_bytes) : 0; }

extern "C" int ddrl_net_forward(ddrl_net* n, const float* const* obs, int n_obs, int B, const float* draw, float* actions,
                                float* logp, float* values, float* pi_out, void* stream) {
  if (!n || B < 0) return DDRL_E_ARG;
  if (!n->params) return DDRL_E_STATE;
  if (B == 0) return DDRL_OK;
  TRY(check_obs(n, obs, n_obs));
  if (!logp || !values || !actions) return DDRL_E_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  TRY(ensure_workspace(n, B, n->ws_train));
  if (n->dirty) TRY(repack(n, s));
  n->cols_obs0 = nullptr;            // the workspace is about to be overwritten
  const int A = n->d.act_dim;
  for (long long r0 = 0; r0 < B; r0 += n->MB) {
    const int mb = (int)std::min<long long>(n->MB, B - r0);
    amax_new_pass(n, s, false);      // every micro-batch rewrites the workspace: amax entries live for one chunk
    TRY(forward_chunk(n, obs, r0, mb, false, s));
    if (n->d.dist == DDRL_DIST_CATEGORICAL) {
      TRY(ddrl_categorical_head(n->logits, n->ldA, draw ? draw + r0 : nullptr, mb, A, actions + r0, logp + r0,
                                pi_out ? pi_out + r0 * A : nullptr, s));
    } else {
      const float* ls = n->params + n->T[n->t_logstd].offset;
      TRY(ddrl_gaussian_head(n->logits, n->ldA, ls, draw ? draw + r0 * A : nullptr, mb, A, actions + r0 * A, logp + r0, s));
      if (pi_out) TRY(copy2d(n->logits, n->ldA, pi_out + r0 * A, A, mb, A, s));
    }
    DDRL_CUDA(cudaMemcpyAsync(values + r0, n->vout, sizeof(float) * mb, cudaMemcpyDeviceToDevice, s));
    for (size_t k = 0; k < n->extra.size(); ++k)     // values is [1 + extras, B]
      DDRL_CUDA(cudaMemcpyAsync(values + (k + 1) * (size_t)B + r0, n->vout_x + k * (size_t)n->MB, sizeof(float) * mb,
                                cudaMemcpyDeviceToDevice, s));
  }
  return DDRL_OK;
}

extern "C" int ddrl_net_encode(ddrl_net* n, const float* const* obs, int n_obs, int B, int tower, float* out, void* stream) {
  if (!n || B < 0 || tower < 0 || tower >= (int)n->towers.size()) return DDRL_E_ARG;
  if (!n->params) return DDRL_E_STATE;
  if (B == 0) return DDRL_OK;
  TRY(check_obs(n, obs, n_obs));
  if (!out) return DDRL_E_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  TRY(ensure_workspace(n, B, n->ws_train));
  if (n->dirty) TRY(repack(n, s));
  n->cols_obs0 = nullptr;            // the workspace is about to be overwritten
  const int F = n->towers[tower].feat;
  for (long long r0 = 0; r0 < B; r0 += n->MB) {
    const int mb = (int)std::min<long long>(n->MB, B - r0);
    amax_new_pass(n, s, false);      // every micro-batch rewrites the workspace: amax entries live for one chunk
    if (n->fuse0) TRY(fused_conv0_fwd(n, obs, r0, mb, false, s, false));
    // towers that borrow tower 0's observation-side im2col matrices need it to have run on this micro-batch
    for (int t = n->towers[tower].borrow_cols ? 0 : tower; t <= tower; ++t) TRY(tower_forward(n, n->towers[t], obs, r0, mb, false, s));
    DDRL_CUDA(cudaMemcpyAsync(out + r0 * F, n->towers[tower].h, sizeof(float) * (size_t)mb * F, cudaMemcpyDeviceToDevice, s));
  }
  return DDRL_OK;
}

namespace ddrl {
// zero the gradients, then per micro-batch: forward (act = data.actions), fused loss, heads and encoders backward; finally
// the packed weight gradients are un-permuted into the reference layout
static int backward_body(ddrl_net* n, const float* const* obs, int B_local, int B_global, const float* actions,
                         const float* old_logp, const float* adv, const float* returns, const float* old_values,
                         const ddrl_ppo_hparams* hp, bool reuse_obs, cudaStream_t s) {
  // zero the flat grads (+ loss tail) and the packed grads: everything below accumulates
  DDRL_CUDA(cudaMemsetAsync(n->grads, 0, sizeof(float) * (size_t)(n->P + 8), s));
  if (n->packed_base) DDRL_CUDA(cudaMemsetAsync(n->packed_base + n->packed_grad_off, 0, n->packed_grad_bytes, s));
  const int A = n->d.act_dim, F = n->d.feat;
  const float invB = 1.0f / (float)B_global;
  float* loss_sums = n->grads + n->P;
  float* stats = hp->ppo_stats ? loss_sums + 3 : nullptr;      // {approx KL, clip fraction} sums in tail slots 3 and 4
  Tower& ta = n->towers[0];
  Tower& tc = n->towers[n->d.shared ? 0 : 1];
  float* aw = n->params + n->T[n->t_aw].offset;
  float* cw = n->params + n->T[n->t_cw].offset;
  for (long long r0 = 0; r0 < B_local; r0 += n->MB) {
    const int mb = (int)std::min<long long>(n->MB, B_local - r0);
    // amax entries live for one micro-batch; the observation-side ones survive while the staged observations do
    amax_new_pass(n, s, reuse_obs);
    TRY(forward_chunk(n, obs, r0, mb, true, s, reuse_obs));
    if (n->d.dist == DDRL_DIST_CATEGORICAL) {
      TRY(ddrl_ppo_loss_categorical_v(n->logits, n->ldA, actions + r0, old_logp + r0, adv + r0, returns + r0, n->vout, mb, A,
                                      invB, hp, n->d.shared, n->dlogits, n->ldA, n->dv, loss_sums,
                                      old_values ? old_values + r0 : nullptr, stats, s));
    } else {
      TRY(ddrl_ppo_loss_gaussian_v(n->logits, n->ldA, n->params + n->T[n->t_logstd].offset, actions + r0 * A, old_logp + r0,
                                   adv + r0, returns + r0, n->vout, mb, A, invB, hp, n->d.shared, n->dlogits, n->ldA, n->dv,
                                   n->grads + n->T[n->t_logstd].offset, loss_sums, old_values ? old_values + r0 : nullptr, stats,
                                   s));
    }
    // heads backward (nn/actor.py:91 actor_linear, nn/critic.py:21 critic_linear)
    TRY(skinny_wgrad(n->dlogits, n->ldA, ta.h, F, mb, A, F, n->grads + n->T[n->t_aw].offset, n->grads + n->T[n->t_ab].offset, s));
    TRY(skinny_wgrad(n->dv, 1, tc.h, F, mb, 1, F, n->grads + n->T[n->t_cw].offset, n->grads + n->T[n->t_cb].offset, s));
    TRY(skinny_dgrad(n->dlogits, n->ldA, aw, mb, A, F, ta.dh, F, 0, s));
    TRY(skinny_dgrad(n->dv, 1, cw, mb, 1, F, tc.dh, F, n->d.shared ? 1 : 0, s));
    // extra value heads (nn/ppo.py:99-107): returns row k+1, loss added to the value-loss sum, gradient into the shared feature
    for (size_t k = 0; k < n->extra.size(); ++k) {
      const ddrl_net::ExtraCritic& x = n->extra[k];
      if (!x.in_loss) continue;
      float* dvx = n->dv_x + k * (size_t)n->MB;
      TRY(ddrl_value_loss(returns + (k + 1) * (size_t)B_local + r0, n->vout_x + k * (size_t)n->MB, mb, invB, hp, n->d.shared, dvx,
                          loss_sums, s));
      TRY(skinny_wgrad(dvx, 1, tc.h, F, mb, 1, F, x.dw, x.db, s));
      TRY(skinny_dgrad(dvx, 1, x.w, mb, 1, F, tc.dh, F, 1, s));
    }
    for (auto& t : n->towers) TRY(tower_backward(n, t, obs, r0, mb, s));
    if (n->fuse0) TRY(fused_conv0_bwd(n, mb, s));
  }
  // packed weight grads -> reference layout
  if (n->cap.active && n->cap.seg > 0) TRY(n->unprep_seg[n->cap.seg].launch("prep_unpack_kernel", s));   // earlier segments: at their cuts
  else if (prep_fused(n) && n->prep_ready) TRY(n->unprep.launch("prep_unpack_kernel", s));
  else TRY(unpack_emit(n, s));
  return DDRL_OK;
}
}  // namespace ddrl

// seg < 0: the whole pass.  seg >= 0: segment `seg` only (seg 0 validates, prepares and -- when the pass is not replayable as
// a graph chain -- runs everything and reports one segment).
static int backward_impl(ddrl_net* n, const float* const* obs, int n_obs, int B_local, int B_global, const float* actions,
                         const float* old_logp, const float* adv, const float* returns, const float* old_values,
                         const ddrl_ppo_hparams* hp, int obs_unchanged, int seg, int* nseg_out, cudaStream_t s) {
  if (!n || !hp || B_local < 0 || B_global < B_local || B_global < 1) return DDRL_E_ARG;
  if (B_local > 0 && !value_clip_ok(hp, old_values)) return DDRL_E_ARG;
  if (!n->params || !n->grads) return DDRL_E_STATE;
  if (nseg_out) *nseg_out = 1;
  if (B_local == 0) {
    if (seg > 0) return DDRL_E_ARG;
    DDRL_CUDA(cudaMemsetAsync(n->grads, 0, sizeof(float) * (size_t)(n->P + 8), s));
    if (n->packed_base) DDRL_CUDA(cudaMemsetAsync(n->packed_base + n->packed_grad_off, 0, n->packed_grad_bytes, s));
    return DDRL_OK;
  }
  TRY(check_obs(n, obs, n_obs));
  if (!actions || !old_logp || !adv || !returns) return DDRL_E_ARG;
  const std::string key = graph_key("bwd", {obs[0], n_obs > 1 ? obs[1] : nullptr, n_obs > 2 ? obs[2] : nullptr, actions, old_logp,
                                            adv, returns, old_values, n->params, n->grads, n->ws.base},
                                    {B_local, B_global}, hp, sizeof(*hp));
  auto launch_seg = [&](ddrl_net::GraphEntry* e, int k) {
    const int pre = (int)e->pre_execs.size();
    if (k < 0 || k > pre) return (int)DDRL_E_ARG;
    DDRL_CUDA(cudaGraphLaunch(k < pre ? e->pre_execs[k] : e->exec, s));
    g_launches += k < pre ? e->pre_launches[k] : e->launches;
    return (int)DDRL_OK;
  };
  if (seg > 0) {
    // later segments of the chain segment 0 of this very call sequence launched
    for (auto& g : n->graphs)
      if (g.key == key) {
        if (nseg_out) *nseg_out = (int)g.pre_execs.size() + 1;
        return launch_seg(&g, seg);
      }
    return DDRL_E_STATE;
  }
  const char* ws_before = n->ws.base;
  TRY(ensure_workspace(n, B_local, true));
  if (n->dirty) TRY(repack(n, s));
  const bool single = B_local <= n->MB;
  const bool reuse_obs = obs_unchanged && single && ws_before == n->ws.base && n->cols_obs0 == obs[0] && n->cols_rows == B_local;
  n->cols_obs0 = single ? obs[0] : nullptr;
  n->cols_rows = single ? B_local : -1;
  // iterations 2..10 of one learn call: same launches, same pointers -> one chain of graph launches
  if (reuse_obs && n->extra.empty() && graphs_enabled(n)) {
    ddrl_net::GraphEntry* e = nullptr;
    TRY(run_graphed(n, key, s, [&](cudaStream_t cs) {
      return backward_body(n, obs, B_local, B_global, actions, old_logp, adv, returns, old_values, hp, true, cs);
    }, seg < 0 ? nullptr : &e));
    if (seg < 0 || !e) return DDRL_OK;             // launched whole / capture failed: the body already ran on the stream
    if (nseg_out) *nseg_out = (int)e->pre_execs.size() + 1;
    return launch_seg(e, 0);
  }
  return backward_body(n, obs, B_local, B_global, actions, old_logp, adv, returns, old_values, hp, reuse_obs, s);
}

extern "C" int ddrl_net_backward(ddrl_net* n, const float* const* obs, int n_obs, int B_local, int B_global,
                                 const float* actions, const float* old_logp, const float* adv, const float* returns,
                                 const ddrl_ppo_hparams* hp, int obs_unchanged, void* stream) {
  return backward_impl(n, obs, n_obs, B_local, B_global, actions, old_logp, adv, returns, nullptr, hp, obs_unchanged, -1, nullptr,
                       (cudaStream_t)stream);
}

extern "C" int ddrl_net_backward_v(ddrl_net* n, const float* const* obs, int n_obs, int B_local, int B_global,
                                   const float* actions, const float* old_logp, const float* adv, const float* returns,
                                   const float* old_values, const ddrl_ppo_hparams* hp, int obs_unchanged, void* stream) {
  return backward_impl(n, obs, n_obs, B_local, B_global, actions, old_logp, adv, returns, old_values, hp, obs_unchanged, -1,
                       nullptr, (cudaStream_t)stream);
}

extern "C" int ddrl_net_backward_segment(ddrl_net* n, const float* const* obs, int n_obs, int B_local, int B_global,
                                         const float* actions, const float* old_logp, const float* adv, const float* returns,
                                         const ddrl_ppo_hparams* hp, int obs_unchanged, int segment, int* n_segments,
                                         void* stream) {
  if (segment < 0 || !n_segments) return DDRL_E_ARG;
  return backward_impl(n, obs, n_obs, B_local, B_global, actions, old_logp, adv, returns, nullptr, hp, obs_unchanged, segment,
                       n_segments, (cudaStream_t)stream);
}

// One minibatch step: new rows at the addresses of an earlier call.  The observations are always restaged (reuse_obs = false),
// so the pass depends on no staging left by an earlier call; the staged observations it leaves belong to no full-batch call.
extern "C" int ddrl_net_backward_minibatch_v(ddrl_net* n, const float* const* obs, int n_obs, int B_local, int B_global,
                                             const float* actions, const float* old_logp, const float* adv, const float* returns,
                                             const float* old_values, const ddrl_ppo_hparams* hp, void* stream) {
  if (!n || !hp || B_local < 0 || B_global < B_local || B_global < 1) return DDRL_E_ARG;
  if (B_local > 0 && !value_clip_ok(hp, old_values)) return DDRL_E_ARG;
  if (!n->params || !n->grads) return DDRL_E_STATE;
  cudaStream_t s = (cudaStream_t)stream;
  if (B_local == 0) {
    DDRL_CUDA(cudaMemsetAsync(n->grads, 0, sizeof(float) * (size_t)(n->P + 8), s));
    if (n->packed_base) DDRL_CUDA(cudaMemsetAsync(n->packed_base + n->packed_grad_off, 0, n->packed_grad_bytes, s));
    return DDRL_OK;
  }
  TRY(check_obs(n, obs, n_obs));
  if (!actions || !old_logp || !adv || !returns) return DDRL_E_ARG;
  TRY(ensure_workspace(n, B_local, true));
  if (n->dirty) TRY(repack(n, s));
  n->cols_obs0 = nullptr;            // a later ddrl_net_backward(obs_unchanged) restages
  n->cols_rows = -1;
  auto body = [&](cudaStream_t cs) {
    return backward_body(n, obs, B_local, B_global, actions, old_logp, adv, returns, old_values, hp, false, cs);
  };
  if (B_local > n->MB || !n->extra.empty() || !graphs_enabled(n) || n->mb_graphs_off) return body(s);
  const std::string key = graph_key("bwd_mb", {obs[0], n_obs > 1 ? obs[1] : nullptr, n_obs > 2 ? obs[2] : nullptr, actions,
                                               old_logp, adv, returns, old_values, n->params, n->grads, n->ws.base},
                                    {B_local, B_global}, hp, sizeof(*hp));
  if (std::find(n->mb_seen.begin(), n->mb_seen.end(), key) == n->mb_seen.end()) {
    if (n->mb_seen.size() >= 16) n->mb_seen.erase(n->mb_seen.begin());
    n->mb_seen.push_back(key);
    return body(s);
  }
  return run_graphed(n, key, s, body, nullptr, &n->mb_graphs_off);
}

extern "C" int ddrl_net_backward_minibatch(ddrl_net* n, const float* const* obs, int n_obs, int B_local, int B_global,
                                           const float* actions, const float* old_logp, const float* adv, const float* returns,
                                           const ddrl_ppo_hparams* hp, void* stream) {
  return ddrl_net_backward_minibatch_v(n, obs, n_obs, B_local, B_global, actions, old_logp, adv, returns, nullptr, hp, stream);
}

// backward segment after which the gradient of parameter tensor `index` is final in the flat gradient buffer
extern "C" int ddrl_net_tensor_segment(const ddrl_net* n, int index) {
  if (!n || index < 0 || index >= (int)n->T.size()) return DDRL_E_ARG;
  if (index == n->t_aw || index == n->t_ab || index == n->t_cw || index == n->t_cb || index == n->t_logstd) return 0;
  for (auto& t : n->towers)
    for (auto& l : t.L)
      if (l.w_t == index || l.b_t == index) return l.seg;
  return n->n_bwd_seg - 1;
}

// debugging aid (not part of the public header): copies workspace buffer `idx` of tower `tower` to `out`
extern "C" int ddrl_net_debug_buffer(ddrl_net* n, int tower, int idx, float* out, int64_t nfloats, void* stream) {
  if (!n || tower < 0 || tower >= (int)n->towers.size()) return DDRL_E_ARG;
  Tower& t = n->towers[tower];
  const float* src = idx == -1 ? t.h : (idx == -2 ? t.dh : (idx >= 0 && idx < (int)t.buf.size() ? t.buf[idx] : nullptr));
  if (!src) return DDRL_E_ARG;
  DDRL_CUDA(cudaMemcpyAsync(out, src, sizeof(float) * nfloats, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return DDRL_OK;
}

namespace ddrl {
__global__ void finish_losses_kernel(const float* __restrict__ sums, float v_coef, float ent_coef, int stats,
                                     float* __restrict__ out) {
  const float a = sums[0], v = sums[1], e = sums[2];
  out[0] = a + v * v_coef - e * ent_coef;      // nn/ppo.py:108
  out[1] = a; out[2] = v; out[3] = e;
  if (stats) { out[4] = sums[3]; out[5] = sums[4]; }
}
}  // namespace ddrl

namespace ddrl {
static int clip_adam_body(ddrl_net* n, int step, const ddrl_ppo_hparams* hp, float* loss4_out, cudaStream_t s) {
  if (loss4_out) {
    finish_losses_kernel<<<1, 1, 0, s>>>(n->grads + n->P, hp->v_coef, hp->ent_coef, hp->ppo_stats, loss4_out);
    DDRL_LAUNCHED("finish_losses_kernel");
  }
  long long sb[3] = {n->seg_begin[0], n->seg_begin[1], n->seg_begin[2]};
  float lr[2];
  if (n->d.shared) lr[0] = hp->lr;
  else { lr[0] = hp->lr_actor; lr[1] = hp->lr_critic; }
  TRY(clip_adam_launch(n->params, n->grads, n->am, n->av, n->P, sb, lr, n->nseg, step, hp, nullptr, s, n->sumsq_dev));
  TRY(repack(n, s));
  return DDRL_OK;
}
}  // namespace ddrl

extern "C" int ddrl_net_clip_adam(ddrl_net* n, int step, const ddrl_ppo_hparams* hp, float* loss4_out, void* stream) {
  if (!n || !hp || step < 1) return DDRL_E_ARG;
  if (!n->params || !n->grads || !n->am || !n->av) return DDRL_E_STATE;
  cudaStream_t s = (cudaStream_t)stream;
  if (!n->sumsq_dev) DDRL_CUDA(cudaMalloc(&n->sumsq_dev, sizeof(double)));
  // the optimiser step + weight re-preparation (~50 small launches on forked side streams) replays as one graph; only the
  // step-dependent scalars of the clip+Adam node change between replays.  The first step of a net runs on the stream (it
  // also performs the one-time allocations a capture must not contain).
  if (step > 1 && !n->dirty && n->packed_base && graphs_enabled(n)) {
    const std::string key = graph_key("adam", {loss4_out, n->params, n->grads, n->am, n->av}, {}, hp, sizeof(*hp));
    ddrl_net::GraphEntry* e = nullptr;
    TRY(run_graphed(n, key, s, [&](cudaStream_t cs) { return clip_adam_body(n, step, hp, loss4_out, cs); }, &e));
    if (!e) return DDRL_OK;                       // capture failed: the body already ran on the stream
    if (!e->adam_node) {
      size_t cnt = 0;
      DDRL_CUDA(cudaGraphGetNodes(e->graph, nullptr, &cnt));
      std::vector<cudaGraphNode_t> nodes(cnt);
      DDRL_CUDA(cudaGraphGetNodes(e->graph, nodes.data(), &cnt));
      for (cudaGraphNode_t nd : nodes) {
        cudaGraphNodeType ty;
        if (cudaGraphNodeGetType(nd, &ty) != cudaSuccess || ty != cudaGraphNodeTypeKernel) continue;
        cudaKernelNodeParams kp;
        if (cudaGraphKernelNodeGetParams(nd, &kp) == cudaSuccess && kp.func == clip_adam_kernel_func()) { e->adam_node = nd; break; }
      }
      if (!e->adam_node) { n->graphs_off = true; graphs_clear(n); return clip_adam_body(n, step, hp, loss4_out, s); }
    }
    long long sb[3] = {n->seg_begin[0], n->seg_begin[1], n->seg_begin[2]};
    float lr[2];
    if (n->d.shared) lr[0] = hp->lr;
    else { lr[0] = hp->lr_actor; lr[1] = hp->lr_critic; }
    TRY(clip_adam_update_node(e->exec, e->adam_node, sb, lr, n->nseg, step, hp));
    DDRL_CUDA(cudaGraphLaunch(e->exec, s));
    g_launches += e->launches;
    n->dirty = false;
    return DDRL_OK;
  }
  return clip_adam_body(n, step, hp, loss4_out, s);
}

