// Host side of the SiamMask hot path: weight ingest (BN fold, repack, fp16 split), the per-frame
// schedule of kernels (backbone -> depthwise xcorr heads -> mask refine) and the C ABI
// (include/siammask_b200.h).  Reference structure restated here:
//   ResNet.forward / _make_layer          experiments/siammask_sharp/resnet.py:151-227
//   ResDown / ResDownS / UP / MaskCorr    experiments/siammask_sharp/custom.py:12-96
//   DepthCorr                             models/rpn.py:41-72
//   Refine.forward(test=True)             experiments/siammask_sharp/custom.py:131-154
//   Custom.template/track/track_mask/track_refine   custom.py:173-190
#include "../../include/siammask_b200.h"
#include "common.cuh"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <unordered_map>

namespace smk {

namespace {

constexpr float BN_EPS = 1e-5f;
constexpr size_t ALIGN = 256;
inline size_t align_up(size_t x) { return (x + ALIGN - 1) / ALIGN * ALIGN; }

thread_local std::string g_last_error;

struct ConvW {
  ConvGeom g{};
  int cout_pad = 0;
  bool gemm_ok = false;
  std::string conv_key, bn_key;       // bn_key empty -> conv has a bias instead
  // tensor-core weight matrix [cout_pad][w_ld]: columns [0,K) this conv, then optionally a second conv whose
  // output is accumulated into the same tile (the bottleneck's downsample branch, fused with conv3) or a
  // diag(2^e) block that lets the residual tensor ride the MMA pipeline (identity segment).
  ConvGeom g2{};
  std::string conv_key2, bn_key2;
  bool fused2 = false, has_diag = false;
  int w_ld = 0, col2 = 0, col_diag = -1;
  size_t off_beta2 = 0;
  float* beta2 = nullptr;             // beta of the fused form (sum of both branches' shifts)
  size_t off_whi = 0, off_wlo = 0, off_wref = 0, off_alpha = 0, off_beta = 0;
  __half* w_hi = nullptr;
  __half* w_lo = nullptr;
  float* w_ref = nullptr;
  float* alpha = nullptr;             // pow2 de-scaling of the tensor-core weights
  float* beta = nullptr;              // folded BN shift / conv bias
  // static power-of-two activation scales (calibrate()): a tensor is STORED as value * 2^s.  s_in / s_in2 / s_res are
  // the scales of this layer's inputs (first conv, fused second conv, residual), s_out of its output; the weights,
  // alpha and beta in the arena are packed for exactly these values (quantize_layer).
  int s_in = 0, s_in2 = 0, s_res = 0, s_out = 0;
  bool f32_out = false;               // output leaves as fp32 (heads, refine inputs): s_out stays 0
  std::vector<std::string> cat_keys;  // non-empty: Cout-concatenation of these layers (one GEMM for all conv_search branches)
  std::string src_in, src_in2, src_res;   // producer tensor names, recorded by the calibration pass
  std::vector<double> shift, shift2;      // unscaled folded shifts (host), kept so the layer can be re-quantized
};

constexpr const char* kSearchCat = "heads.conv_search_cat";

struct F32T {                         // fp32 NHWC tensor (refine stage)
  float* p = nullptr;
  int B = 0, H = 0, W = 0, C = 0;
};

struct ProfRec {
  std::string name, cat;
  double flops = 0, bytes = 0;
  cudaEvent_t e0 = nullptr, e1 = nullptr;
};

struct Arena {
  uint8_t* base = nullptr;
  size_t cap = 0, off = 0, peak = 0;
  bool measure = false;
  void reset() { off = 0; }
  void* alloc(size_t bytes) {
    off = align_up(off);
    void* p = base + off;
    off += bytes;
    peak = std::max(peak, off);
    if (!measure) SMK_CHECK(off <= cap, "workspace arena exhausted");
    return p;
  }
};

// One execution lane: its own workspace, stream set and cached per-step tensors.  A batch of >= 2 * kLaneMinB streams
// is split over two lanes that run concurrently (streams are independent): the persistent GEMM kernels of one lane
// fill the SMs the other lane's kernels leave idle in their last wave and in the low-occupancy refine tail.
struct Lane {
  Arena search, refine;
  std::map<std::string, Act> named;            // p0, p1, p2, search, corr_* of the lane's last track
  cudaStream_t own = nullptr;                  // the lane's main stream (lane 0 runs on the caller's stream in the device-pointer API)
  cudaStream_t aux[3] = {nullptr, nullptr, nullptr};
  int cap_B = 0;                               // largest batch this lane's arenas were sized for
};
constexpr int kMaxLanes = 2;                   // 3 or 4 lanes measured slower than 2 (DESIGN.md §5)
constexpr int kLaneMinB = 8;                   // a lane gets at least this many streams (below 2 x 8: one lane)

}  // namespace

class Engine {
 public:
  explicit Engine(const sm_config& cfg);
  ~Engine() { release(); }

  void load_weights(const sm_tensor_desc* t, int n);
  void adopt_weights();
  void calibrate(int B, const float* z, const float* x, cudaStream_t st);
  int status();
  void weight_blob(void** p, size_t* bytes) { *p = blob_; *bytes = blob_bytes_; }

  void do_template(int slot0, int B, const float* z, cudaStream_t st);
  void do_track(int slot0, int B, const float* x, float* cls, float* loc, float* mask, int flags, cudaStream_t st);
  void do_refine(int B, const int32_t* pos, float* out, cudaStream_t st);
  void set_graphs(bool on) { use_graphs_ = on; }
  void track_host(int slot0, int B, const float* xh, float* clsh, float* loch, const int32_t* posh, float* maskh,
                  cudaStream_t st);
  int track_host_async(int slot0, int B, const float* xh, float* clsh, float* loch, const int32_t* posh, float* maskh,
                       cudaStream_t st);
  void host_wait(int ticket);
  // whole frame: track(+mask) -> on-device score/box selection -> refine at the selected position
  struct StepIO {
    const float* x = nullptr;            // device or (host path) staged input
    const double* tsz = nullptr;         // [B][2] target_sz * scale_x
    const float* anchors = nullptr;      // device [A*R*R][4]
    const float* window = nullptr;       // device [A*R*R]
    double penalty_k = 0, window_influence = 0;
    int flags = 0;
    float* cls = nullptr; float* loc = nullptr; float* mask = nullptr;   // device outputs (mask: raw 3969-ch head)
    int32_t* best = nullptr; int32_t* pos = nullptr; float* rec = nullptr;
    float* refine = nullptr;             // [B][127*127] or null
    float* mask_col = nullptr;           // [B][3969] = mask[b, :, dy, dx] or null
  };
  void do_step(int slot0, int B, const StepIO& io, cudaStream_t st);
  int step_host_async(int slot0, int B, const sm_step_io& io, cudaStream_t st);
  void do_export(const char* what, float* out, int64_t* shape4, cudaStream_t st);

  void set_profiling(bool on) { profiling_ = on; }
  std::string profile_dump();
  int64_t launches() const { return launches_; }
  size_t bytes() const { return total_bytes_; }
  const sm_config& cfg() const { return cfg_; }

 private:
  // ---- construction
  void construct(const sm_config& cfg);
  ConvW& add_layer(const std::string& conv_key, const std::string& bn_key, ConvGeom g);
  void build_layer_table();
  void assign_blob_layout();
  size_t measure_arena(int B, int S, bool search);
  size_t refine_arena_bytes(int B) const;
  // ---- packing
  void fold_layer(ConvW& L, const std::map<std::string, const sm_tensor_desc*>& sd, uint8_t* host);
  void quantize_layer(ConvW& L, uint8_t* host);
  void quantize_stem(uint8_t* host);
  void write_scale_table(uint8_t* host);
  void read_scale_table(const uint8_t* host);
  void upload_blob();
  int tscale(const std::string& name) const {
    auto it = tscale_.find(name);
    return it == tscale_.end() ? 0 : it->second;
  }
  void note_tensor(const Act& a, const std::string& name, cudaStream_t st);
  // ---- schedule
  Act alloc_act(Arena& ar, int B, int H, int W, int C);
  F32T alloc_f32(Arena& ar, int B, int H, int W, int C);
  Act conv(const Act& in, const ConvW& L, bool relu, const Act* res, Arena& ar, cudaStream_t st,
           const Act* in2 = nullptr);
  void conv_into(const Act& in, const ConvW& L, Epilogue ep, cudaStream_t st, const Act* res = nullptr,
                 const Act* in2 = nullptr);
  F32T conv_f32(const Act& in, const ConvW& L, bool relu, Arena& ar, cudaStream_t st);
  Act backbone(const float* x, int B, int S, Arena& ar, bool keep, cudaStream_t st);
  F32T small(const F32T& a, const F32T* b, int Ho, const ConvW& L, bool relu, float* out_override, Arena& ar,
             cudaStream_t st);
  const ConvW& L(const std::string& k) const {
    auto it = layers_.find(k);
    SMK_CHECK(it != layers_.end(), "unknown layer " + k);
    return it->second;
  }
  const int* updown_map(int out, int in) const {
    auto it = maps_.find(out * 1000 + in);
    SMK_CHECK(it != maps_.end(), "no upsample map");
    return it->second;
  }

  sm_config cfg_;
  bool exact_;
  int num_sms_ = 148;
  int R_ = 0;                          // response size (score_size)
  std::map<std::string, ConvW> layers_;
  std::vector<std::string> layer_order_;
  size_t off_deconv_w_ = 0, off_deconv_b_ = 0, off_ones_ = 0;
  size_t off_stem_whi_ = 0, off_stem_wlo_ = 0, off_stem_alpha_ = 0;
  __half* stem_whi_ = nullptr;
  __half* stem_wlo_ = nullptr;
  float* stem_alpha_ = nullptr;
  float* deconv_w_ = nullptr;
  float* deconv_b_ = nullptr;
  float* ones_ = nullptr;              // alpha for the SIMT reference path (weights unscaled)
  uint8_t* blob_ = nullptr;
  size_t blob_bytes_ = 0;
  bool weights_ready_ = false;
  std::vector<uint8_t> host_blob_;                       // host image of the arena (kept: re-quantization after calibrate)
  size_t off_scales_ = 0;
  std::map<std::string, int> tscale_;                    // scales of tensors that are not conv outputs: stem, corr_*
  int* ovf_flag_ = nullptr;                              // device: set when an activation left fp16's range
  // calibration pass: producer name per activation buffer, max |value| per tensor name
  bool calibrating_ = false;
  std::unordered_map<const void*, std::string> tensor_name_;
  std::vector<std::string> absmax_names_;
  float* absmax_dev_ = nullptr;
  static constexpr int kAbsmaxSlots = 256;

  Arena templ_arena_;
  Lane lanes_[kMaxLanes];
  Lane* cur_ = &lanes_[0];             // lane whose schedule is being enqueued
  int n_lanes_ = 1;                    // kMaxLanes, capped by max_batch / kLaneMinB
  int split_n_ = 1;                    // how the last track divided its batch: lane l got streams
  int split_off_[kMaxLanes + 1] = {0, 0, 0};   //   [split_off_[l], split_off_[l + 1])
  // per-slot template caches: [branch][slot][5][5][256] split planes, and zf for export
  __half* kcache_hi_ = nullptr;
  __half* kcache_lo_ = nullptr;
  int n_branches_ = 2;
  // host-path staging
  // two sets (ping-pong) so the H2D of step k+1 and the D2H of step k overlap the compute of the other step
  float* stage_x_[2] = {nullptr, nullptr};
  float* stage_cls_[2] = {nullptr, nullptr};
  float* stage_loc_[2] = {nullptr, nullptr};
  float* stage_mask_[2] = {nullptr, nullptr};
  int32_t* stage_pos_[2] = {nullptr, nullptr};
  double* stage_tsz_[2] = {nullptr, nullptr};
  float* stage_rec_[2] = {nullptr, nullptr};
  int32_t* stage_best_[2] = {nullptr, nullptr};
  float* stage_maskcol_[2] = {nullptr, nullptr};
  float* mask_raw_ = nullptr;          // [max_batch][3969][R][R] raw mask-head output of the host-buffer step (lazy)
  void step_lane(int slot0, int B, const StepIO& io, cudaStream_t st);
  void release();
  cudaStream_t h2d_stream_ = nullptr, d2h_stream_ = nullptr;
  cudaEvent_t h2d_done_[2] = {nullptr, nullptr}, compute_done_[2] = {nullptr, nullptr}, d2h_done_[2] = {nullptr, nullptr};
  bool set_busy_[2] = {false, false};
  uint64_t host_calls_ = 0;
  int* maps_dev_ = nullptr;
  std::map<int, const int*> maps_;

  // state of the last track (Custom.feature / .search / .corr_feature, custom.py:182-184)
  Act zf_;                             // template feature of the last sm_template (export)
  bool have_zf_ = false;
  int last_B_ = 0;
  bool have_mask_feats_ = false;

  int64_t launches_ = 0;
  size_t total_bytes_ = 0;
  bool measuring_ = false;

  // L2-aware traversal: for every activation buffer, which end was touched last (+1 = highest rows, -1 = lowest).
  // A GEMM whose largest input was last touched at its high end walks its M tiles in reverse, and vice versa, so
  // each layer starts on the ~100 MB of its input that are still in L2 instead of re-streaming all of it from HBM.
  std::unordered_map<const void*, int> last_end_;
  int end_of(const Act& a) const {
    auto it = last_end_.find(a.hi);
    return it == last_end_.end() ? +1 : it->second;      // the non-GEMM kernels write front to back
  }

  // CUDA-graph replay of a whole track / refine call (launch-bound small batches).  A call signature seen once
  // runs eagerly, the second time it is captured (all work, including the auxiliary-stream branches, hangs off
  // the caller's stream) and from then on replayed; the host-side bookkeeping of the call is restored with it.
  struct GraphEntry {
    int seen = 0;
    cudaGraphExec_t exec = nullptr;
    std::map<std::string, Act> named[kMaxLanes];
    int split_n = 1;
    int split_off[kMaxLanes + 1] = {0, 0, 0};
    int last_B = 0;
    bool have_mask_feats = false;
    int64_t launches = 0;
  };
  bool use_graphs_ = false;
  std::map<std::vector<uint64_t>, GraphEntry> graphs_;
  void track_impl(int slot0, int B, const float* x, float* cls, float* loc, float* mask, int flags, cudaStream_t st);
  void track_lane(int slot0, int B, const float* x, float* cls, float* loc, float* mask, int flags, cudaStream_t st);
  void refine_impl(int B, const int32_t* pos, float* out, cudaStream_t st);
  void refine_lane(int B, const int32_t* pos, float* out, cudaStream_t st);
  bool defer_join_ = false;            // host-buffer path: lane 1 stays forked between its track and its refine
  bool lane1_forked_ = false;          // lanes 1.. are forked from the caller's stream and not joined back yet
  // host-buffer path with two lanes: both lanes run on their own streams and are never joined into the caller's
  // stream — each only waits for its inputs, the D2H waits for both — so consecutive steps of the two lanes slide
  // against each other.  The next stream-ordered entry point (template / track / refine / export) joins them.
  bool lanes_dirty_ = false;
  cudaEvent_t lane_done_[2][kMaxLanes] = {};   // [staging set][lane]
  void join_lanes(cudaStream_t st) {
    if (!lanes_dirty_) return;
    for (int l = 0; l < n_lanes_; ++l) order_after(lanes_[l].own, st);
    lanes_dirty_ = false;
  }
  static int lanes_for(int n_lanes, int B) { return std::max(1, std::min(n_lanes, B / kLaneMinB)); }
  static int chunk(int B, int nl, int l) { return B / nl + (l < B % nl ? 1 : 0); }
  void split_batch(int B) {
    // per-launch profiling (bench.py roofline) times every layer as ONE launch over the whole batch: per-kernel
    // durations are not defined while two lanes interleave, and half-batch launches timed back to back would charge
    // each kernel the idle last wave that the other lane fills in the real schedule
    split_n_ = (profiling_ || calibrating_) ? 1 : lanes_for(n_lanes_, B);
    split_off_[0] = 0;
    for (int l = 0; l < split_n_; ++l) {
      split_off_[l + 1] = split_off_[l] + chunk(B, split_n_, l);
      SMK_CHECK(chunk(B, split_n_, l) <= lanes_[l].cap_B, "lane workspace too small for this batch");
    }
  }
  void fork_lanes(cudaStream_t st) {
    if (split_n_ < 2 || !concurrent() || lane1_forked_) return;
    for (int l = 1; l < split_n_; ++l) order_after(st, lanes_[l].own);
    lane1_forked_ = true;
  }
  void join_forked(cudaStream_t st) {
    if (!lane1_forked_) return;
    for (int l = 1; l < n_lanes_; ++l) order_after(lanes_[l].own, st);
    lane1_forked_ = false;
  }
  // if a schedule throws half way (arena exhausted, launch error), leave the lanes joined and lane 0 current
  struct LaneGuard {
    Engine* e; cudaStream_t st; bool armed = true;
    ~LaneGuard() {
      if (!armed) return;
      e->cur_ = &e->lanes_[0];
      e->defer_join_ = false;
      try { e->join_forked(st); } catch (...) {}
    }
  };
  template <typename F>
  void run_with_graph(const std::vector<uint64_t>& key, cudaStream_t st, F&& body) {
    if (!use_graphs_ || profiling_ || calibrating_) { body(); return; }
    GraphEntry& ge = graphs_[key];
    if (ge.exec != nullptr) {
      SMK_CUDA(cudaGraphLaunch(ge.exec, st));
      for (int l = 0; l < kMaxLanes; ++l)
        for (auto& kv : ge.named[l]) lanes_[l].named[kv.first] = kv.second;
      split_n_ = ge.split_n;
      for (int l = 0; l <= kMaxLanes; ++l) split_off_[l] = ge.split_off[l];
      last_B_ = ge.last_B;
      have_mask_feats_ = ge.have_mask_feats;
      launches_ += ge.launches;
      return;
    }
    if (ge.seen++ == 0) { body(); return; }          // first sight: eager (also warms function attributes)
    const int64_t l0 = launches_;
    cudaGraph_t graph = nullptr;
    SMK_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
    try {
      body();
    } catch (...) {
      cudaStreamEndCapture(st, &graph);
      if (graph) cudaGraphDestroy(graph);
      throw;
    }
    SMK_CUDA(cudaStreamEndCapture(st, &graph));
    SMK_CUDA(cudaGraphInstantiate(&ge.exec, graph, 0));
    SMK_CUDA(cudaGraphDestroy(graph));
    for (int l = 0; l < kMaxLanes; ++l) ge.named[l] = lanes_[l].named;
    ge.split_n = split_n_;
    for (int l = 0; l <= kMaxLanes; ++l) ge.split_off[l] = split_off_[l];
    ge.last_B = last_B_;
    ge.have_mask_feats = have_mask_feats_;
    ge.launches = launches_ - l0;
    SMK_CUDA(cudaGraphLaunch(ge.exec, st));
  }

  // independent sub-graphs (the three correlation heads; the refine stage's v-branches) run on auxiliary
  // streams forked from / joined back into the caller's stream with events
  static constexpr int kAux = 3;
  std::vector<cudaEvent_t> sync_events_;
  size_t sync_next_ = 0;
  cudaEvent_t next_sync_event() {
    cudaEvent_t e = sync_events_[sync_next_];
    sync_next_ = (sync_next_ + 1) % sync_events_.size();
    return e;
  }
  bool concurrent() const { return !profiling_ && !calibrating_; }
  // make `to` wait for everything enqueued on `from` so far
  void order_after(cudaStream_t from, cudaStream_t to) {
    if (from == to) return;
    cudaEvent_t e = next_sync_event();
    SMK_CUDA(cudaEventRecord(e, from));
    SMK_CUDA(cudaStreamWaitEvent(to, e, 0));
  }

  // optional per-launch CUDA-event timing (bench.py roofline): records (name, category, flops, bytes, e0, e1)
  bool profiling_ = false;
  std::vector<ProfRec> prof_;
  std::vector<cudaEvent_t> event_pool_;
  cudaEvent_t get_event() {
    if (!event_pool_.empty()) { cudaEvent_t e = event_pool_.back(); event_pool_.pop_back(); return e; }
    cudaEvent_t e;
    SMK_CUDA(cudaEventCreate(&e));
    return e;
  }
  struct Scope {
    Engine* eng; cudaStream_t st; size_t idx; bool on;
    Scope(Engine* e, const std::string& name, const char* cat, double flops, double bytes, cudaStream_t s)
        : eng(e), st(s), idx(0), on(e->profiling_ && !e->measuring_) {
      if (!on) return;
      ProfRec r;
      r.name = name; r.cat = cat; r.flops = flops; r.bytes = bytes;
      r.e0 = eng->get_event(); r.e1 = eng->get_event();
      cudaEventRecord(r.e0, st);
      idx = eng->prof_.size();
      eng->prof_.push_back(r);
    }
    ~Scope() { if (on) cudaEventRecord(eng->prof_[idx].e1, st); }
  };
};

// ================================================================================================
// construction

ConvW& Engine::add_layer(const std::string& conv_key, const std::string& bn_key, ConvGeom g) {
  ConvW w;
  w.g = g;
  w.conv_key = conv_key;
  w.bn_key = bn_key;
  w.gemm_ok = gemm_conv_supported(g);
  w.cout_pad = w.gemm_ok ? gemm_cout_pad(g.Cout) : g.Cout;
  w.w_ld = g.KH * g.KW * g.Cin;
  layer_order_.push_back(conv_key);
  return layers_[conv_key] = w;
}

void Engine::build_layer_table() {
  const std::string F = "features.features.";
  add_layer(F + "conv1", F + "bn1", {3, 64, 7, 7, 2, 0, 1});
  struct LayerSpec { const char* name; int planes, blocks, stride, dilation; };
  const LayerSpec specs[3] = {{"layer1", 64, 3, 1, 1}, {"layer2", 128, 4, 2, 1}, {"layer3", 256, 6, 1, 2}};
  int inplanes = 64;
  for (const auto& sp : specs) {
    for (int i = 0; i < sp.blocks; ++i) {
      const std::string P = F + sp.name + "." + std::to_string(i) + ".";
      int stride = 1, dil = sp.dilation;
      if (i == 0) {                       // _make_layer, resnet.py:184-215
        stride = sp.stride;
        dil = sp.dilation > 1 ? sp.dilation / 2 : 1;
        ConvGeom ds;
        if (sp.stride == 1 && sp.dilation == 1) ds = {inplanes, sp.planes * 4, 1, 1, 1, 0, 1};
        else if (sp.dilation > 1) ds = {inplanes, sp.planes * 4, 3, 3, sp.stride, sp.dilation / 2, sp.dilation / 2};
        else ds = {inplanes, sp.planes * 4, 3, 3, sp.stride, 0, 1};
        add_layer(P + "downsample.0", P + "downsample.1", ds);
      }
      const int pad = dil > 1 ? dil : 2 - stride;   // Bottleneck.__init__, resnet.py:66-70
      add_layer(P + "conv1", P + "bn1", {inplanes, sp.planes, 1, 1, 1, 0, 1});
      add_layer(P + "conv2", P + "bn2", {sp.planes, sp.planes, 3, 3, stride, pad, dil});
      ConvW& c3 = add_layer(P + "conv3", P + "bn3", {sp.planes, sp.planes * 4, 1, 1, 1, 0, 1});
      if (i == 0) {                       // out = relu(bn3(conv3(t)) + bn_ds(conv_ds(x))): one GEMM, K = K3 + Kds
        const ConvW& ds = layers_[P + "downsample.0"];
        c3.fused2 = true;
        c3.g2 = ds.g;
        c3.conv_key2 = ds.conv_key;
        c3.bn_key2 = ds.bn_key;
      } else {                            // out = relu(bn3(conv3(t)) + x): residual via the identity segment
        c3.has_diag = true;
      }
      inplanes = sp.planes * 4;
    }
  }
  add_layer("features.downsample.downsample.0", "features.downsample.downsample.1", {1024, 256, 1, 1, 1, 0, 1});
  std::vector<std::pair<std::string, int>> heads = {{"rpn_model.cls.", 2 * cfg_.anchor_num},
                                                    {"rpn_model.loc.", 4 * cfg_.anchor_num}};
  if (cfg_.with_mask) heads.push_back({"mask_model.mask.", 63 * 63});
  n_branches_ = (int)heads.size();
  for (auto& h : heads) {
    add_layer(h.first + "conv_kernel.0", h.first + "conv_kernel.1", {256, 256, 3, 3, 1, 0, 1});
    add_layer(h.first + "conv_search.0", h.first + "conv_search.1", {256, 256, 3, 3, 1, 0, 1});
    add_layer(h.first + "head.0", h.first + "head.1", {256, 256, 1, 1, 1, 0, 1});
    add_layer(h.first + "head.3", "", {256, h.second, 1, 1, 1, 0, 1});
  }
  {
    // DepthCorr.conv_search of every branch reads the same search feature (models/rpn.py:63-67): one GEMM with the
    // branches' output channels concatenated (N = 256 x branches) instead of one launch and one pass over xf per branch
    ConvW& cat = add_layer(kSearchCat, "", {256, 256 * n_branches_, 3, 3, 1, 0, 1});
    for (auto& h : heads) cat.cat_keys.push_back(h.first + "conv_search.0");
  }
  if (cfg_.with_mask) {
    const std::string R = "refine_model.";
    auto c3 = [&](const std::string& k, int ci, int co) { add_layer(R + k, "", {ci, co, 3, 3, 1, 1, 1}); };
    c3("v0.0", 64, 16);  c3("v0.2", 16, 4);
    c3("v1.0", 256, 64); c3("v1.2", 64, 16);
    c3("v2.0", 512, 128); c3("v2.2", 128, 32);
    c3("h2.0", 32, 32);  c3("h2.2", 32, 32);
    c3("h1.0", 16, 16);  c3("h1.2", 16, 16);
    c3("h0.0", 4, 4);    c3("h0.2", 4, 4);
    c3("post0", 32, 16); c3("post1", 16, 4); c3("post2", 4, 1);
  }
}

void Engine::assign_blob_layout() {
  size_t off = 0;
  for (const auto& k : layer_order_) {
    ConvW& w = layers_[k];
    const size_t K = (size_t)w.g.KH * w.g.KW * w.g.Cin;
    w.w_ld = (int)K;
    if (w.fused2) { w.col2 = w.w_ld; w.w_ld += w.g2.KH * w.g2.KW * w.g2.Cin; }
    if (w.has_diag) { w.col_diag = w.w_ld; w.w_ld += w.g.Cout; }
    if (w.gemm_ok) {
      w.off_whi = off; off = align_up(off + (size_t)w.cout_pad * w.w_ld * sizeof(__half));
      w.off_wlo = off; off = align_up(off + (size_t)w.cout_pad * w.w_ld * sizeof(__half));
    }
    w.off_beta2 = off; off = align_up(off + (size_t)w.cout_pad * sizeof(float));
    w.off_wref = off;  off = align_up(off + K * w.g.Cout * sizeof(float));
    w.off_alpha = off; off = align_up(off + (size_t)w.cout_pad * sizeof(float));
    w.off_beta = off;  off = align_up(off + (size_t)w.cout_pad * sizeof(float));
  }
  off_ones_ = off; off = align_up(off + 4096 * sizeof(float));
  off_stem_whi_ = off; off = align_up(off + 64 * 192 * sizeof(__half));
  off_stem_wlo_ = off; off = align_up(off + 64 * 192 * sizeof(__half));
  off_stem_alpha_ = off; off = align_up(off + 64 * sizeof(float));
  if (cfg_.with_mask) {
    off_deconv_w_ = off; off = align_up(off + (size_t)256 * 7200 * sizeof(float));
    off_deconv_b_ = off; off = align_up(off + 32 * sizeof(float));
  }
  off_scales_ = off; off = align_up(off + (layer_order_.size() * 4 + 4) * sizeof(int32_t));
  blob_bytes_ = off;
}

Engine::Engine(const sm_config& cfg) : cfg_(cfg), exact_(cfg.precision == SM_PRECISION_EXACT) {
  try {
    construct(cfg);
  } catch (...) {
    release();           // a half-built engine must not leak its device allocations, streams and events
    throw;
  }
}

void Engine::construct(const sm_config& cfg) {
  SMK_CHECK(cfg.search_size >= 127 && (cfg.search_size - 127) % 8 == 0, "search_size must be 127 + 8k");
  SMK_CHECK(cfg.max_batch >= 1 && cfg.num_slots >= cfg.max_batch, "need num_slots >= max_batch >= 1");
  SMK_CHECK(cfg.anchor_num >= 1, "anchor_num");
  int dev = 0;
  SMK_CUDA(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  SMK_CUDA(cudaGetDeviceProperties(&prop, dev));
  SMK_CHECK(prop.major == 10, "siammask_b200 kernels are built for sm_100a only (found sm_" +
                                  std::to_string(prop.major) + std::to_string(prop.minor) + ")");
  num_sms_ = prop.multiProcessorCount;
  R_ = (cfg.search_size - 127) / 8 + 1 + 8;   // utils/tracker_config.py:23,46 with base_size 8

  build_layer_table();
  assign_blob_layout();
  SMK_CUDA(cudaMalloc(&blob_, blob_bytes_));
  SMK_CUDA(cudaMalloc(&ovf_flag_, sizeof(int)));
  SMK_CUDA(cudaMemset(ovf_flag_, 0, sizeof(int)));
  for (auto& kv : layers_) {
    ConvW& w = kv.second;
    if (w.gemm_ok) {
      w.w_hi = reinterpret_cast<__half*>(blob_ + w.off_whi);
      w.w_lo = reinterpret_cast<__half*>(blob_ + w.off_wlo);
    }
    w.w_ref = reinterpret_cast<float*>(blob_ + w.off_wref);
    w.alpha = reinterpret_cast<float*>(blob_ + w.off_alpha);
    w.beta = reinterpret_cast<float*>(blob_ + w.off_beta);
    w.beta2 = reinterpret_cast<float*>(blob_ + w.off_beta2);
  }
  ones_ = reinterpret_cast<float*>(blob_ + off_ones_);
  stem_whi_ = reinterpret_cast<__half*>(blob_ + off_stem_whi_);
  stem_wlo_ = reinterpret_cast<__half*>(blob_ + off_stem_wlo_);
  stem_alpha_ = reinterpret_cast<float*>(blob_ + off_stem_alpha_);
  if (cfg_.with_mask) {
    deconv_w_ = reinterpret_cast<float*>(blob_ + off_deconv_w_);
    deconv_b_ = reinterpret_cast<float*>(blob_ + off_deconv_b_);
  }

  // workspace sizes: dry-run the schedule with a measuring arena
  n_lanes_ = lanes_for(kMaxLanes, cfg.max_batch);
  // the largest chunk each lane can be handed over all batch sizes this engine accepts (lane 0: the whole batch,
  // when profiling)
  lanes_[0].cap_B = cfg.max_batch;
  for (int B = 1; B <= cfg.max_batch; ++B) {
    const int nl = lanes_for(n_lanes_, B);
    for (int l = 0; l < nl; ++l) lanes_[l].cap_B = std::max(lanes_[l].cap_B, chunk(B, nl, l));
  }
  templ_arena_.cap = measure_arena(cfg.max_batch, 127, false);
  SMK_CUDA(cudaMalloc(&templ_arena_.base, templ_arena_.cap));
  for (int l = 0; l < n_lanes_; ++l) {
    Lane& ln = lanes_[l];
    ln.search.cap = measure_arena(ln.cap_B, cfg.search_size, true);
    SMK_CUDA(cudaMalloc(&ln.search.base, ln.search.cap));
    if (cfg_.with_mask) {
      ln.refine.cap = refine_arena_bytes(ln.cap_B);
      SMK_CUDA(cudaMalloc(&ln.refine.base, ln.refine.cap));
    }
    for (int i = 0; i < kAux; ++i) SMK_CUDA(cudaStreamCreateWithFlags(&ln.aux[i], cudaStreamNonBlocking));
    SMK_CUDA(cudaStreamCreateWithFlags(&ln.own, cudaStreamNonBlocking));
  }
  const size_t kc = (size_t)n_branches_ * cfg.num_slots * 25 * 256;
  SMK_CUDA(cudaMalloc(&kcache_hi_, kc * sizeof(__half)));
  SMK_CUDA(cudaMalloc(&kcache_lo_, kc * sizeof(__half)));
  SMK_CUDA(cudaMemset(kcache_hi_, 0, kc * sizeof(__half)));
  SMK_CUDA(cudaMemset(kcache_lo_, 0, kc * sizeof(__half)));

  const size_t B = cfg.max_batch, S = cfg.search_size, A = cfg.anchor_num;
  for (int i = 0; i < 2; ++i) {
    SMK_CUDA(cudaMalloc(&stage_x_[i], B * 3 * S * S * sizeof(float)));
    SMK_CUDA(cudaMalloc(&stage_cls_[i], B * 2 * A * R_ * R_ * sizeof(float)));
    SMK_CUDA(cudaMalloc(&stage_loc_[i], B * 4 * A * R_ * R_ * sizeof(float)));
    SMK_CUDA(cudaMalloc(&stage_mask_[i], B * 127 * 127 * sizeof(float)));
    SMK_CUDA(cudaMalloc(&stage_pos_[i], B * 2 * sizeof(int32_t)));
    SMK_CUDA(cudaMalloc(&stage_tsz_[i], B * 2 * sizeof(double)));
    SMK_CUDA(cudaMalloc(&stage_rec_[i], B * 8 * sizeof(float)));
    SMK_CUDA(cudaMalloc(&stage_best_[i], B * sizeof(int32_t)));
    if (cfg_.with_mask) SMK_CUDA(cudaMalloc(&stage_maskcol_[i], B * 3969 * sizeof(float)));
    SMK_CUDA(cudaEventCreateWithFlags(&h2d_done_[i], cudaEventDisableTiming));
    SMK_CUDA(cudaEventCreateWithFlags(&compute_done_[i], cudaEventDisableTiming));
    SMK_CUDA(cudaEventCreateWithFlags(&d2h_done_[i], cudaEventDisableTiming));
    for (int l = 0; l < kMaxLanes; ++l) SMK_CUDA(cudaEventCreateWithFlags(&lane_done_[i][l], cudaEventDisableTiming));
  }
  SMK_CUDA(cudaStreamCreateWithFlags(&h2d_stream_, cudaStreamNonBlocking));
  SMK_CUDA(cudaStreamCreateWithFlags(&d2h_stream_, cudaStreamNonBlocking));

  // nearest-upsample index tables (custom.py:150-152) + identity tables
  const int pairs[6][2] = {{31, 15}, {61, 31}, {127, 61}, {15, 15}, {31, 31}, {61, 61}};
  std::vector<int> all;
  std::vector<size_t> offs;
  for (auto& pr : pairs) {
    offs.push_back(all.size());
    auto t = nearest_index_table(pr[0], pr[1]);
    all.insert(all.end(), t.begin(), t.end());
  }
  SMK_CUDA(cudaMalloc(&maps_dev_, all.size() * sizeof(int)));
  SMK_CUDA(cudaMemcpy(maps_dev_, all.data(), all.size() * sizeof(int), cudaMemcpyHostToDevice));
  for (int i = 0; i < 6; ++i) maps_[pairs[i][0] * 1000 + pairs[i][1]] = maps_dev_ + offs[i];
  sync_events_.resize(64);
  for (auto& e : sync_events_) SMK_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));

  size_t lane_bytes = 0;
  for (auto& ln : lanes_) lane_bytes += ln.search.cap + ln.refine.cap;
  total_bytes_ = blob_bytes_ + templ_arena_.cap + lane_bytes + 2 * kc * sizeof(__half) +
                 2 * (B * 3 * S * S + B * 6 * A * R_ * R_ + B * 127 * 127) * sizeof(float);
}

void Engine::release() {
  cudaFree(blob_);
  cudaFree(templ_arena_.base);
  for (auto& ln : lanes_) {
    cudaFree(ln.search.base);
    cudaFree(ln.refine.base);
    for (int i = 0; i < kAux; ++i) if (ln.aux[i]) cudaStreamDestroy(ln.aux[i]);
    if (ln.own) cudaStreamDestroy(ln.own);
  }
  cudaFree(kcache_hi_);
  cudaFree(kcache_lo_);
  for (int i = 0; i < 2; ++i) {
    cudaFree(stage_x_[i]); cudaFree(stage_cls_[i]); cudaFree(stage_loc_[i]); cudaFree(stage_mask_[i]); cudaFree(stage_pos_[i]);
    cudaFree(stage_tsz_[i]); cudaFree(stage_rec_[i]); cudaFree(stage_best_[i]); cudaFree(stage_maskcol_[i]);
    if (h2d_done_[i]) cudaEventDestroy(h2d_done_[i]);
    if (compute_done_[i]) cudaEventDestroy(compute_done_[i]);
    if (d2h_done_[i]) cudaEventDestroy(d2h_done_[i]);
    for (int l = 0; l < kMaxLanes; ++l) if (lane_done_[i][l]) cudaEventDestroy(lane_done_[i][l]);
  }
  if (h2d_stream_) cudaStreamDestroy(h2d_stream_);
  if (d2h_stream_) cudaStreamDestroy(d2h_stream_);
  cudaFree(maps_dev_);
  cudaFree(mask_raw_);
  cudaFree(ovf_flag_);
  cudaFree(absmax_dev_);
  for (auto e : sync_events_) cudaEventDestroy(e);
  for (auto e : event_pool_) cudaEventDestroy(e);
  for (auto& kv : graphs_) if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
}

// every allocation refine_lane makes, in its order (the window sizes 15 / 31 / 61 / 127 are fixed by custom.py:131-152)
size_t Engine::refine_arena_bytes(int B) const {
  size_t off = 0;
  auto add = [&](size_t bytes) { off = align_up(off) + bytes; };
  auto act = [&](int hw, int c) { add((size_t)B * hw * hw * c * sizeof(__half)); if (exact_) add((size_t)B * hw * hw * c * sizeof(__half)); };
  auto f32 = [&](int hw, int c) { add((size_t)B * hw * hw * c * sizeof(float)); };
  act(15, 512); act(15, 128); f32(15, 32);          // c2, v2.0, v2.2
  act(31, 256); act(31, 64); f32(31, 16);           // c1, v1.0, v1.2
  act(61, 64); f32(61, 16); f32(61, 4);             // c0, v0.0, v0.2
  add((size_t)B * 256 * sizeof(float)); f32(15, 32);// p3, deconv
  f32(15, 32); f32(15, 32); f32(31, 16);            // h2.0, h2.2, post0
  f32(31, 16); f32(31, 16); f32(61, 4);             // h1.0, h1.2, post1
  f32(61, 4); f32(61, 4);                           // h0.0, h0.2 (post2 writes the caller's buffer)
  return align_up(off + (1u << 16));
}

size_t Engine::measure_arena(int B, int S, bool search) {
  Arena ar;
  ar.measure = true;
  measuring_ = true;
  Act xf = backbone(nullptr, B, S, ar, search, nullptr);
  if (search) {
    // heads: conv_search, corr, head.0 per branch
    alloc_act(ar, B, xf.H - 2, xf.W - 2, 256 * n_branches_);      // conv_search of all branches (one GEMM or one each)
    for (int br = 0; br < n_branches_; ++br) {
      alloc_act(ar, B, R_, R_, 256);
      alloc_act(ar, B, R_, R_, 256);
    }
  }
  measuring_ = false;
  cur_->named.clear();
  return align_up(ar.peak + (1u << 20));
}

// ================================================================================================
// weight ingest

namespace {
const float* find_tensor(const std::map<std::string, const sm_tensor_desc*>& sd, const std::string& name,
                         size_t expect_numel) {
  auto it = sd.find(name);
  SMK_CHECK(it != sd.end(), "checkpoint is missing tensor '" + name + "'");
  size_t n = 1;
  for (int i = 0; i < it->second->ndim; ++i) n *= (size_t)it->second->shape[i];
  SMK_CHECK(n == expect_numel, "tensor '" + name + "' has " + std::to_string(n) + " elements, expected " +
                                   std::to_string(expect_numel));
  return it->second->data;
}
}  // namespace

namespace {
// eval-mode BatchNorm folded to y = conv(x, w) * scale + shift (or the conv's own bias when there is no BN)
void fold_affine(const std::map<std::string, const sm_tensor_desc*>& sd, const std::string& conv_key,
                 const std::string& bn_key, int cout, std::vector<double>& scale, std::vector<double>& shift) {
  scale.assign(cout, 1.0);
  shift.assign(cout, 0.0);
  if (!bn_key.empty()) {
    const float* gm = find_tensor(sd, bn_key + ".weight", cout);
    const float* bt = find_tensor(sd, bn_key + ".bias", cout);
    const float* mu = find_tensor(sd, bn_key + ".running_mean", cout);
    const float* var = find_tensor(sd, bn_key + ".running_var", cout);
    for (int n = 0; n < cout; ++n) {
      scale[n] = (double)gm[n] / std::sqrt((double)var[n] + (double)BN_EPS);
      shift[n] = (double)bt[n] - (double)mu[n] * scale[n];
    }
  } else {
    const float* b = find_tensor(sd, conv_key + ".bias", cout);
    for (int n = 0; n < cout; ++n) shift[n] = b[n];
  }
}
}  // namespace

// Step 1 of the ingest: BN folding (float64) into fp32 weights [K][Cout] (`w_ref`, also the SIMT backend's operand)
// and unscaled shifts.  Needs the checkpoint; everything after this works from the host image alone.
void Engine::fold_layer(ConvW& L, const std::map<std::string, const sm_tensor_desc*>& sd, uint8_t* host) {
  const ConvGeom& g = L.g;
  const size_t K = (size_t)g.KH * g.KW * g.Cin;
  if (!L.cat_keys.empty()) {          // concatenation of already folded layers along Cout
    float* w_cat = reinterpret_cast<float*>(host + L.off_wref);
    L.shift.assign(g.Cout, 0.0);
    int n0 = 0;
    for (const auto& key : L.cat_keys) {
      const ConvW& src = layers_.at(key);
      SMK_CHECK(src.g.Cin == g.Cin && src.g.KH == g.KH && !src.shift.empty(), "concatenated layers must share their geometry");
      const float* ws = reinterpret_cast<const float*>(host + src.off_wref);
      for (size_t k = 0; k < K; ++k)
        for (int n = 0; n < src.g.Cout; ++n) w_cat[k * g.Cout + n0 + n] = ws[k * src.g.Cout + n];
      for (int n = 0; n < src.g.Cout; ++n) L.shift[n0 + n] = src.shift[n];
      n0 += src.g.Cout;
    }
    return;
  }
  const float* w = find_tensor(sd, L.conv_key + ".weight", K * g.Cout);   // OIHW
  std::vector<double> scale;
  fold_affine(sd, L.conv_key, L.bn_key, g.Cout, scale, L.shift);
  float* w_ref = reinterpret_cast<float*>(host + L.off_wref);
  const int HW = g.KH * g.KW;
  for (int n = 0; n < g.Cout; ++n)
    for (int c = 0; c < g.Cin; ++c)
      for (int t = 0; t < HW; ++t)
        w_ref[((size_t)t * g.Cin + c) * g.Cout + n] = (float)((double)w[((size_t)n * g.Cin + c) * HW + t] * scale[n]);
}

// Step 2: tensor-core operands for the layer's current activation scales.  With inputs stored as a * 2^s_in (a2 * 2^s_in2,
// r * 2^s_res) the accumulator of output channel n is 2^(e_n + s_in) * sum(w a) when
//   * the first conv's weights are scaled by 2^e_n (per-channel, keeps hi AND lo fp16 parts normal),
//   * the fused second conv's by 2^(e_n + s_in - s_in2),
//   * the residual's diag entry is 2^(e_n + s_in - s_res);
// the epilogue's alpha = 2^(s_out - s_in - e_n) and beta = shift * 2^s_out then store the output at 2^s_out.
void Engine::quantize_layer(ConvW& L, uint8_t* host) {
  const ConvGeom& g = L.g;
  const size_t K = (size_t)g.KH * g.KW * g.Cin;
  const size_t K2 = L.fused2 ? (size_t)L.g2.KH * L.g2.KW * L.g2.Cin : 0;
  const float* w_ref = reinterpret_cast<const float*>(host + L.off_wref);
  const ConvW* L2 = L.fused2 ? &layers_.at(L.conv_key2) : nullptr;
  const float* w_ref2 = L2 ? reinterpret_cast<const float*>(host + L2->off_wref) : nullptr;
  float* alpha = reinterpret_cast<float*>(host + L.off_alpha);
  float* beta = reinterpret_cast<float*>(host + L.off_beta);
  float* beta2 = reinterpret_cast<float*>(host + L.off_beta2);
  __half* w_hi = L.gemm_ok ? reinterpret_cast<__half*>(host + L.off_whi) : nullptr;
  __half* w_lo = L.gemm_ok ? reinterpret_cast<__half*>(host + L.off_wlo) : nullptr;
  for (int n = 0; n < L.cout_pad; ++n) { alpha[n] = 0.f; beta[n] = 0.f; beta2[n] = 0.f; }
  const size_t ld = (size_t)L.w_ld;
  const int d2 = L.s_in - L.s_in2;                  // relative scale of the fused second conv's weights
  for (int n = 0; n < g.Cout; ++n) {
    float amax = 0.f;
    for (size_t k = 0; k < K; ++k) amax = std::max(amax, std::fabs(w_ref[k * g.Cout + n]));
    for (size_t k = 0; k < K2; ++k) amax = std::max(amax, std::fabs(std::ldexp(w_ref2[k * g.Cout + n], d2)));
    beta[n] = (float)std::ldexp(L.shift[n], L.s_out);
    beta2[n] = (float)std::ldexp(L.shift[n] + (L2 ? L2->shift[n] : 0.0), L.s_out);
    alpha[n] = std::ldexp(1.f, L.s_out - L.s_in);
    if (!L.gemm_ok) continue;
    // per-output-channel power-of-two scaling keeps hi AND lo fp16 parts in the normal range; |e| <= 14, and with a
    // residual the diag entry 2^(e + s_in - s_res) must itself be a normal fp16
    int e = 0;
    if (amax > 0.f) e = (int)std::floor(std::log2(16384.0 / (double)amax));
    e = std::max(-14, std::min(14, e));
    if (L.has_diag) {
      const int d = L.s_in - L.s_res;
      e = std::max(-14 - d, std::min(14 - d, e));
      SMK_CHECK(e >= -24 && e <= 24, "activation scales of a residual block are too far apart");
    }
    alpha[n] = std::ldexp(1.f, L.s_out - L.s_in - e);
    __half* rh = w_hi + (size_t)n * ld;
    __half* rl = w_lo + (size_t)n * ld;
    for (size_t k = 0; k < K; ++k) {
      const float fw = std::ldexp(w_ref[k * g.Cout + n], e);
      const __half h = __float2half_rn(fw);
      rh[k] = h;
      rl[k] = __float2half_rn(fw - __half2float(h));
    }
    for (size_t k = 0; k < K2; ++k) {
      const float fw = std::ldexp(w_ref2[k * g.Cout + n], e + d2);
      const __half h = __float2half_rn(fw);
      rh[L.col2 + k] = h;
      rl[L.col2 + k] = __float2half_rn(fw - __half2float(h));
    }
    if (L.has_diag) rh[L.col_diag + n] = __float2half_rn(std::ldexp(1.f, e + L.s_in - L.s_res));   // rest stays 0
  }
}

// tensor-core stem: [64][192] K-major, k = (r*7+s)*3 + c — exactly the row index of the folded w_ref; output at 2^s
void Engine::quantize_stem(uint8_t* host) {
  ConvW& stem = layers_["features.features.conv1"];
  const int s_out = tscale("stem");
  stem.s_out = s_out;
  const float* wref = reinterpret_cast<const float*>(host + stem.off_wref);
  __half* sh = reinterpret_cast<__half*>(host + off_stem_whi_);
  __half* sl = reinterpret_cast<__half*>(host + off_stem_wlo_);
  float* sa = reinterpret_cast<float*>(host + off_stem_alpha_);
  float* sb = reinterpret_cast<float*>(host + stem.off_beta);
  for (int n = 0; n < 64; ++n) {
    float amax = 0.f;
    for (int k = 0; k < 147; ++k) amax = std::max(amax, std::fabs(wref[(size_t)k * 64 + n]));
    int e = amax > 0.f ? (int)std::floor(std::log2(16384.0 / (double)amax)) : 0;
    e = std::max(-14, std::min(14, e));
    sa[n] = std::ldexp(1.f, s_out - e);
    sb[n] = (float)std::ldexp(stem.shift[n], s_out);
    for (int k = 0; k < 147; ++k) {
      const float fw = std::ldexp(wref[(size_t)k * 64 + n], e);
      const __half h = __float2half_rn(fw);
      sh[n * 192 + k] = h;
      sl[n * 192 + k] = __float2half_rn(fw - __half2float(h));
    }
  }
}

// the scales travel with the arena (NCCL broadcast / packed-weight file): 4 ints per layer + the named tensors
static const char* kNamedTensors[4] = {"stem", "corr_cls", "corr_loc", "corr_mask"};
void Engine::write_scale_table(uint8_t* host) {
  int32_t* t = reinterpret_cast<int32_t*>(host + off_scales_);
  size_t i = 0;
  for (const auto& k : layer_order_) {
    const ConvW& w = layers_[k];
    t[i++] = w.s_in; t[i++] = w.s_in2; t[i++] = w.s_res; t[i++] = w.s_out;
  }
  for (const char* nm : kNamedTensors) t[i++] = tscale(nm);
}
void Engine::read_scale_table(const uint8_t* host) {
  const int32_t* t = reinterpret_cast<const int32_t*>(host + off_scales_);
  size_t i = 0;
  for (const auto& k : layer_order_) {
    ConvW& w = layers_[k];
    w.s_in = t[i++]; w.s_in2 = t[i++]; w.s_res = t[i++]; w.s_out = t[i++];
  }
  for (const char* nm : kNamedTensors) tscale_[nm] = t[i++];
}

void Engine::upload_blob() {
  write_scale_table(host_blob_.data());
  SMK_CUDA(cudaMemcpy(blob_, host_blob_.data(), blob_bytes_, cudaMemcpyHostToDevice));
}

// weights arrived by broadcast / from a packed file: take the activation scales from the arena
void Engine::adopt_weights() {
  std::vector<uint8_t> tbl(blob_bytes_ - off_scales_);
  SMK_CUDA(cudaMemcpy(tbl.data(), blob_ + off_scales_, tbl.size(), cudaMemcpyDeviceToHost));
  read_scale_table(tbl.data() - off_scales_);
  host_blob_.clear();                 // no host image: calibrate() needs load_weights on this engine
  weights_ready_ = true;
}

void Engine::load_weights(const sm_tensor_desc* t, int n) {
  std::map<std::string, const sm_tensor_desc*> sd;
  for (int i = 0; i < n; ++i) {
    SMK_CHECK(t[i].name != nullptr && t[i].data != nullptr, "null tensor descriptor");
    std::string name = t[i].name;
    if (name.rfind("module.", 0) == 0) name = name.substr(7);   // utils/load_helper.py:22-27
    sd[name] = &t[i];
  }
  host_blob_.assign(blob_bytes_, 0);
  uint8_t* host = host_blob_.data();
  tscale_.clear();
  for (const auto& k : layer_order_) {
    ConvW& w = layers_[k];
    w.s_in = w.s_in2 = w.s_res = w.s_out = 0;
    fold_layer(w, sd, host);
  }
  for (const auto& k : layer_order_) quantize_layer(layers_[k], host);
  float* ones = reinterpret_cast<float*>(host + off_ones_);
  for (int i = 0; i < 4096; ++i) ones[i] = 1.f;
  quantize_stem(host);
  if (cfg_.with_mask) {
    // ConvTranspose2d weight (Cin=256, Cout=32, 15, 15) -> [k][(y*15+x)*32 + co]
    const float* dw = find_tensor(sd, "refine_model.deconv.weight", (size_t)256 * 32 * 225);
    const float* db = find_tensor(sd, "refine_model.deconv.bias", 32);
    float* wd = reinterpret_cast<float*>(host + off_deconv_w_);
    for (int k = 0; k < 256; ++k)
      for (int co = 0; co < 32; ++co)
        for (int p = 0; p < 225; ++p) wd[(size_t)k * 7200 + p * 32 + co] = dw[((size_t)k * 32 + co) * 225 + p];
    std::memcpy(host + off_deconv_b_, db, 32 * sizeof(float));
  }
  upload_blob();
  weights_ready_ = true;
}


// Static activation scales.  Every activation lives in HBM as two fp16 planes of value * 2^s (hi + lo, 22 significant
// bits) — fp16's exponent range is narrow: |value * 2^s| must stay below 65504, and `lo` keeps full precision only
// while `hi` stays above ~2^-3.  calibrate() runs the whole path (template, track_mask incl. the mask head, refine) on
// a sample batch, measures max |value| of every tensor and picks s per tensor so that the maximum sits near 2^10
// (64x headroom above the sample, full lo precision down to 2^-13 of the maximum); the weights / alpha / beta of every
// layer are then re-quantized for those scales (quantize_layer).  conv+BN is linear and ReLU / max-pool / crops commute
// with a positive scale, so this costs nothing at run time.  Without calibration all scales are 0: fine for networks
// whose activations are O(1)..O(10^3) (BN-normalised checkpoints); the overflow flag (status()) tells otherwise.
void Engine::calibrate(int B, const float* z, const float* x, cudaStream_t st) {
  SMK_CHECK(weights_ready_ && !host_blob_.empty(), "calibrate() needs weights loaded through sm_engine_load_weights on this engine");
  SMK_CHECK(cfg_.backend == SM_BACKEND_TENSOR, "calibrate() applies to the tensor-core backend");
  SMK_CHECK(B >= 1 && B <= cfg_.max_batch && z != nullptr && x != nullptr, "calibration batch");
  join_lanes(st);
  const size_t A = cfg_.anchor_num, RR = (size_t)R_ * R_;
  float *cls = nullptr, *loc = nullptr, *mask = nullptr, *ref = nullptr;
  int32_t* pos = nullptr;
  struct Tmp { std::vector<void*> p; ~Tmp() { for (void* q : p) cudaFree(q); } } tmp;
  auto dalloc = [&](size_t bytes) { void* q = nullptr; SMK_CUDA(cudaMalloc(&q, bytes)); tmp.p.push_back(q); return q; };
  cls = static_cast<float*>(dalloc(B * 2 * A * RR * sizeof(float)));
  loc = static_cast<float*>(dalloc(B * 4 * A * RR * sizeof(float)));
  if (cfg_.with_mask) {
    mask = static_cast<float*>(dalloc((size_t)B * 3969 * RR * sizeof(float)));
    ref = static_cast<float*>(dalloc((size_t)B * 127 * 127 * sizeof(float)));
    pos = static_cast<int32_t*>(dalloc((size_t)B * 2 * sizeof(int32_t)));
    std::vector<int32_t> hp((size_t)B * 2, R_ / 2);
    SMK_CUDA(cudaMemcpy(pos, hp.data(), hp.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
  }
  if (absmax_dev_ == nullptr) SMK_CUDA(cudaMalloc(&absmax_dev_, kAbsmaxSlots * sizeof(float)));
  for (auto& kv : graphs_) if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
  graphs_.clear();                                   // replayed graphs bake the old scale factors into kernel arguments

  auto scale_of = [&](const std::string& name) -> int {
    auto it = layers_.find(name);
    return it != layers_.end() ? it->second.s_out : tscale(name);
  };
  auto set_scale = [&](const std::string& name, int v) {
    auto it = layers_.find(name);
    if (it != layers_.end()) it->second.s_out = it->second.f32_out ? 0 : v;
    else tscale_[name] = v;
  };
  auto rewire_and_upload = [&]() {
    {
      // the per-branch conv_search layers (used when only some branches run) mirror the concatenated one
      const ConvW& cat = layers_.at(kSearchCat);
      if (!cat.src_in.empty())
        for (const auto& k : cat.cat_keys) {
          ConvW& w = layers_.at(k);
          w.src_in = cat.src_in;
          w.s_out = cat.s_out;
        }
    }
    for (auto& kv : layers_) {
      ConvW& w = kv.second;
      if (!w.src_in.empty()) w.s_in = scale_of(w.src_in);
      if (!w.src_in2.empty()) w.s_in2 = scale_of(w.src_in2);
      if (!w.src_res.empty()) w.s_res = scale_of(w.src_res);
    }
    for (const auto& k : layer_order_) quantize_layer(layers_[k], host_blob_.data());
    quantize_stem(host_blob_.data());
    upload_blob();
  };

  bool settled = false;
  for (int iter = 0; iter < 12 && !settled; ++iter) {
    SMK_CUDA(cudaMemsetAsync(absmax_dev_, 0, kAbsmaxSlots * sizeof(float), st));
    SMK_CUDA(cudaMemsetAsync(ovf_flag_, 0, sizeof(int), st));
    struct Guard { Engine* e; ~Guard() { e->calibrating_ = false; e->tensor_name_.clear(); } } guard{this};
    calibrating_ = true;
    absmax_names_.clear();
    tensor_name_.clear();
    do_template(0, B, z, st);
    if (cfg_.with_mask) {
      do_track(0, B, x, cls, loc, mask, SM_TRACK_MASK_FEATURES | SM_TRACK_MASK_HEAD, st);
      do_refine(B, pos, ref, st);
    } else {
      do_track(0, B, x, cls, loc, nullptr, 0, st);
    }
    SMK_CUDA(cudaStreamSynchronize(st));
    calibrating_ = false;
    std::vector<float> mx(absmax_names_.size());
    SMK_CUDA(cudaMemcpy(mx.data(), absmax_dev_, mx.size() * sizeof(float), cudaMemcpyDeviceToHost));
    bool any_inf = false, any_zero = false;
    for (float v : mx) {
      if (!(v <= 65504.f)) any_inf = true;
      if (v == 0.f) any_zero = true;
    }
    if (any_inf || (any_zero && iter < 8)) {
      // out of range somewhere: everything downstream of it is meaningless — move ALL scales and look again
      const int step = any_inf ? -10 : +10;
      for (size_t i = 0; i < mx.size(); ++i) set_scale(absmax_names_[i], scale_of(absmax_names_[i]) + step);
      rewire_and_upload();
      continue;
    }
    settled = true;
    for (size_t i = 0; i < mx.size(); ++i) {
      if (mx[i] == 0.f) continue;
      const int cur = scale_of(absmax_names_[i]);
      // stored maximum already in [2^8, 2^12]: leave the tensor alone (a well-scaled checkpoint keeps s = 0 and its
      // results bit for bit); otherwise re-target the stored maximum to ~2^10
      if (mx[i] >= 256.f && mx[i] <= 4096.f) continue;
      int want = cur + (int)std::lround(std::log2(1024.0 / (double)mx[i]));
      want = std::max(-60, std::min(60, want));
      const auto it = layers_.find(absmax_names_[i]);
      if (it != layers_.end() && it->second.f32_out) want = 0;
      if (want != cur) { set_scale(absmax_names_[i], want); settled = false; }
    }
    if (!settled) rewire_and_upload();
  }
  SMK_CHECK(settled, "calibrate(): activation scales did not settle (non-finite network outputs?)");
}

int Engine::status() {
  int v = 0;
  SMK_CUDA(cudaDeviceSynchronize());
  SMK_CUDA(cudaMemcpy(&v, ovf_flag_, sizeof(int), cudaMemcpyDeviceToHost));
  return v;
}

// ================================================================================================
// schedule helpers

Act Engine::alloc_act(Arena& ar, int B, int H, int W, int C) {
  Act a;
  a.B = B; a.H = H; a.W = W; a.C = C;
  a.hi = static_cast<__half*>(ar.alloc(a.numel() * sizeof(__half)));
  a.lo = exact_ ? static_cast<__half*>(ar.alloc(a.numel() * sizeof(__half))) : nullptr;
  return a;
}

F32T Engine::alloc_f32(Arena& ar, int B, int H, int W, int C) {
  F32T t;
  t.B = B; t.H = H; t.W = W; t.C = C;
  t.p = static_cast<float*>(ar.alloc((size_t)B * H * W * C * sizeof(float)));
  return t;
}

void Engine::conv_into(const Act& in, const ConvW& Lw, Epilogue ep, cudaStream_t st, const Act* res,
                       const Act* in2) {
  if (measuring_) return;
  ep.beta = Lw.beta;
  ++launches_;
  const double M = (double)in.B * Lw.g.out_size(in.H) * Lw.g.out_size(in.W);
  double K = (double)Lw.g.KH * Lw.g.KW * Lw.g.Cin;
  const bool tc = cfg_.backend == SM_BACKEND_TENSOR && Lw.gemm_ok;
  SMK_CHECK(in2 == nullptr || (tc && Lw.fused2), "fused second input needs the tensor-core path");
  if (in2 != nullptr) K += (double)Lw.g2.KH * Lw.g2.KW * Lw.g2.Cin;
  if (calibrating_) {
    // record which tensors feed this layer (the scales of a layer's operands are those of their producers)
    ConvW& W = const_cast<ConvW&>(Lw);
    auto name_of = [&](const Act& a) {
      auto it = tensor_name_.find(a.hi);
      return it == tensor_name_.end() ? std::string() : it->second;
    };
    W.src_in = name_of(in);
    W.src_in2 = in2 ? name_of(*in2) : std::string();
    W.src_res = res ? name_of(*res) : std::string();
    W.f32_out = ep.out_mode != OUT_NHWC_SPLIT;
  }
  SMK_CHECK(in.sexp == Lw.s_in && (in2 == nullptr || in2->sexp == Lw.s_in2) && (res == nullptr || res->sexp == Lw.s_res),
            "activation scale mismatch at " + Lw.conv_key + " (weights were packed for other scales: re-run calibrate)");
  SMK_CHECK(ep.out_mode == OUT_NHWC_SPLIT || Lw.s_out == 0, "fp32 outputs are unscaled");
  if (ep.out_mode == OUT_NHWC_SPLIT) ep.ovf = ovf_flag_;
  Scope sc(this, Lw.conv_key, tc ? "conv_gemm" : "conv_simt", 2.0 * M * K * Lw.g.Cout,
           4.0 * ((double)in.numel() + (in2 ? (double)in2->numel() : 0.0) + M * Lw.g.Cout * (res ? 2 : 1) +
                  K * Lw.g.Cout), st);
  if (tc) {
    ep.alpha = Lw.alpha;
    // start where the biggest input was touched last
    const Act* big = &in;
    if (in2 != nullptr && in2->numel() > big->numel()) big = in2;
    if (res != nullptr && res->numel() > big->numel()) big = res;
    // bottleneck conv2 (3x3 / s1 / p1, 64 or 128 channels): resident-patch kernel, walks its tiles front to back
    const bool use_patch = in2 == nullptr && res == nullptr &&
                           ep.out_mode == OUT_NHWC_SPLIT && patch_conv_supported(in, Lw.g);
    const bool reverse = !use_patch && end_of(*big) > 0;
    const int now_end = reverse ? -1 : +1;
    last_end_[in.hi] = now_end;
    if (in2 != nullptr) last_end_[in2->hi] = now_end;
    if (res != nullptr) last_end_[res->hi] = now_end;
    if (ep.out_mode == OUT_NHWC_SPLIT) last_end_[ep.out_hi] = now_end;
    GemmInput gi[2] = {{in, Lw.g, 0}, {in, Lw.g, 0}};
    int nconv = 1;
    const Act* ident = nullptr;
    if (in2 != nullptr) {
      gi[1] = {*in2, Lw.g2, Lw.col2};
      nconv = 2;
      ep.beta = Lw.beta2;
    } else if (res != nullptr) {
      if (Lw.has_diag) ident = res;                                  // residual through the MMA pipeline
      else { ep.res_hi = res->hi; ep.res_lo = res->lo; }             // epilogue-side add
    }
    if (use_patch)
      launch_conv3x3_patch(in, Lw.g, Lw.w_hi, Lw.w_lo, Lw.w_ld, ep, exact_ ? 2 : 1, num_sms_, st);
    else
      launch_gemm_multi(gi, nconv, ident, Lw.col_diag, Lw.w_hi, Lw.w_lo, Lw.cout_pad, Lw.w_ld, ep, exact_ ? 2 : 1,
                        num_sms_, st, reverse);
  } else {
    SMK_CHECK(Lw.s_in == 0 && Lw.s_out == 0, "the SIMT backend runs unscaled activations only");
    ep.alpha = ones_;
    if (res != nullptr) { ep.res_hi = res->hi; ep.res_lo = res->lo; }
    launch_ref_conv(in, Lw.g, Lw.w_ref, ep, st);
  }
}

// calibration pass: remember which tensor lives in this buffer and fold its max |value| into the tensor's slot
void Engine::note_tensor(const Act& a, const std::string& name, cudaStream_t st) {
  if (!calibrating_ || measuring_) return;
  tensor_name_[a.hi] = name;
  size_t slot = 0;
  for (; slot < absmax_names_.size(); ++slot)
    if (absmax_names_[slot] == name) break;
  if (slot == absmax_names_.size()) {
    SMK_CHECK((int)slot < kAbsmaxSlots, "too many calibrated tensors");
    absmax_names_.push_back(name);
  }
  launch_absmax(a, absmax_dev_ + slot, st);
}

Act Engine::conv(const Act& in, const ConvW& Lw, bool relu, const Act* res, Arena& ar, cudaStream_t st,
                 const Act* in2) {
  Act out = alloc_act(ar, in.B, Lw.g.out_size(in.H), Lw.g.out_size(in.W), Lw.g.Cout);
  Epilogue ep;
  ep.relu = relu ? 1 : 0;
  ep.out_mode = OUT_NHWC_SPLIT;
  ep.out_hi = out.hi;
  ep.out_lo = out.lo;
  out.sexp = Lw.s_out;
  conv_into(in, Lw, ep, st, res, in2);
  note_tensor(out, Lw.conv_key, st);
  return out;
}

F32T Engine::conv_f32(const Act& in, const ConvW& Lw, bool relu, Arena& ar, cudaStream_t st) {
  F32T out = alloc_f32(ar, in.B, Lw.g.out_size(in.H), Lw.g.out_size(in.W), Lw.g.Cout);
  Epilogue ep;
  ep.relu = relu ? 1 : 0;
  ep.out_mode = OUT_NHWC_F32;
  ep.out_f32 = out.p;
  conv_into(in, Lw, ep, st);
  return out;
}

// ResDown.forward / forward_all (custom.py:58-66): ResNet (resnet.py:217-227) + ResDownS (custom.py:19-25)
Act Engine::backbone(const float* x, int B, int S, Arena& ar, bool keep, cudaStream_t st) {
  const std::string F = "features.features.";
  const int So = (S - 7) / 2 + 1;
  Act p0 = alloc_act(ar, B, So, So, 64);
  const ConvW& stem = L(F + "conv1");
  if (!measuring_) {
    Scope sc(this, "stem", "stem", 2.0 * B * So * So * 64 * 147, 4.0 * B * (3.0 * S * S + 64.0 * So * So), st);
    if (cfg_.backend == SM_BACKEND_TENSOR)
      launch_stem_tc(x, B, S, stem_whi_, stem_wlo_, stem_alpha_, stem.beta, p0, num_sms_, st, ovf_flag_);
    else launch_stem(x, B, S, stem.w_ref, ones_, stem.beta, p0, st);
    ++launches_;
  }
  p0.sexp = stem.s_out;
  note_tensor(p0, "stem", st);
  const int Sp = (So + 2 - 3) / 2 + 1;
  Act y = alloc_act(ar, B, Sp, Sp, 64);
  y.sexp = p0.sexp;                    // max-pool commutes with a positive scale
  if (calibrating_ && !measuring_) tensor_name_[y.hi] = "stem";
  if (!measuring_) {
    Scope sc(this, "maxpool", "pool", 0, 4.0 * (p0.numel() + y.numel()), st);
    launch_maxpool3s2(p0, y, st);
    ++launches_;
  }
  last_end_[p0.hi] = +1;       // stem and pool write front to back
  last_end_[y.hi] = +1;
  if (keep) cur_->named["p0"] = p0;
  const char* names[3] = {"layer1", "layer2", "layer3"};
  const int blocks[3] = {3, 4, 6};
  for (int l = 0; l < 3; ++l) {
    for (int i = 0; i < blocks[l]; ++i) {
      const std::string P = F + names[l] + "." + std::to_string(i) + ".";
      Act t1 = conv(y, L(P + "conv1"), true, nullptr, ar, st);
      Act t2 = conv(t1, L(P + "conv2"), true, nullptr, ar, st);
      const ConvW& c3 = L(P + "conv3");
      if (i == 0 && cfg_.backend == SM_BACKEND_TENSOR && c3.fused2) {
        y = conv(t2, c3, true, nullptr, ar, st, &y);            // conv3 + downsample branch in one GEMM
      } else {
        Act res = y;
        if (i == 0) res = conv(y, L(P + "downsample.0"), false, nullptr, ar, st);
        y = conv(t2, c3, true, &res, ar, st);
      }
    }
    if (keep) cur_->named[std::string("p") + std::to_string(l + 1)] = y;
  }
  Act xf = conv(y, L("features.downsample.downsample.0"), false, nullptr, ar, st);
  if (xf.W < 20) {   // custom.py:21-24
    Act c = alloc_act(ar, B, xf.H - 8, xf.W - 8, xf.C);
    c.sexp = xf.sexp;
    if (calibrating_ && !measuring_) tensor_name_[c.hi] = tensor_name_[xf.hi];
    if (!measuring_) { launch_crop_center(xf, 4, c, st); ++launches_; }
    xf = c;
  }
  return xf;
}

static const char* kBranch[3] = {"rpn_model.cls.", "rpn_model.loc.", "mask_model.mask."};
static const char* kCorrName[3] = {"corr_cls", "corr_loc", "corr_mask"};

void Engine::do_template(int slot0, int B, const float* z, cudaStream_t st) {
  SMK_CHECK(weights_ready_, "weights not loaded");
  SMK_CHECK(B >= 1 && B <= cfg_.max_batch && slot0 >= 0 && slot0 + B <= cfg_.num_slots, "template batch/slot range");
  join_lanes(st);
  templ_arena_.reset();
  Act zf = backbone(z, B, 127, templ_arena_, false, st);
  SMK_CHECK(zf.H == 7 && zf.W == 7, "template feature must be 7x7");
  zf_ = zf;
  have_zf_ = true;
  for (int br = 0; br < n_branches_; ++br) {
    const ConvW& ck = L(std::string(kBranch[br]) + "conv_kernel.0");
    Epilogue ep;
    ep.relu = 1;
    ep.out_mode = OUT_NHWC_SPLIT;
    const size_t off = ((size_t)br * cfg_.num_slots + slot0) * 25 * 256;
    ep.out_hi = kcache_hi_ + off;
    ep.out_lo = exact_ ? kcache_lo_ + off : nullptr;
    conv_into(zf, ck, ep, st);
    if (calibrating_) {
      Act kc;
      kc.hi = ep.out_hi; kc.lo = ep.out_lo; kc.B = B; kc.H = 5; kc.W = 5; kc.C = 256;
      note_tensor(kc, ck.conv_key, st);
    }
  }
}

void Engine::do_track(int slot0, int B, const float* x, float* cls, float* loc, float* mask, int flags,
                      cudaStream_t st) {
  join_lanes(st);
  const std::vector<uint64_t> key = {1, (uint64_t)slot0, (uint64_t)B, (uint64_t)x, (uint64_t)cls, (uint64_t)loc,
                                     (uint64_t)mask, (uint64_t)flags, (uint64_t)st};
  run_with_graph(key, st, [&] { track_impl(slot0, B, x, cls, loc, mask, flags, st); });
}

void Engine::track_impl(int slot0, int B, const float* x, float* cls, float* loc, float* mask, int flags,
                        cudaStream_t st) {
  SMK_CHECK(weights_ready_, "weights not loaded");
  SMK_CHECK(B >= 1 && B <= cfg_.max_batch && slot0 >= 0 && slot0 + B <= cfg_.num_slots, "track batch/slot range");
  SMK_CHECK(cls != nullptr && loc != nullptr, "cls/loc outputs required");
  const bool want_feats = (flags & SM_TRACK_MASK_FEATURES) != 0;
  const bool want_mask_head = (flags & SM_TRACK_MASK_HEAD) != 0;
  SMK_CHECK(!(want_feats || want_mask_head) || cfg_.with_mask, "engine was built without the mask branch");
  SMK_CHECK(!want_mask_head || mask != nullptr, "mask output buffer required");
  // split the streams over the two lanes; lane 1 forks from / joins back into the caller's stream
  split_batch(B);
  const int nl = split_n_;
  LaneGuard guard{this, st};
  const size_t S = cfg_.search_size, A = cfg_.anchor_num, RR = (size_t)R_ * R_;
  // fork before anything of this call is enqueued on `st`, so the lanes really run side by side
  fork_lanes(st);
  for (int l = nl - 1; l >= 0; --l) {
    cur_ = &lanes_[l];
    const int b0 = split_off_[l], nbat = split_off_[l + 1] - split_off_[l];
    cudaStream_t ls = (l == 0 || !concurrent()) ? st : lanes_[l].own;
    track_lane(slot0 + b0, nbat, x + b0 * 3 * S * S, cls + b0 * 2 * A * RR, loc + b0 * 4 * A * RR,
               mask != nullptr ? mask + (size_t)b0 * 63 * 63 * RR : nullptr, flags, ls);
  }
  cur_ = &lanes_[0];
  guard.armed = false;
  if (!defer_join_) join_forked(st);
  last_B_ = B;
  have_mask_feats_ = want_feats || want_mask_head;
}

void Engine::track_lane(int slot0, int B, const float* x, float* cls, float* loc, float* mask, int flags,
                        cudaStream_t st) {
  const bool want_feats = (flags & SM_TRACK_MASK_FEATURES) != 0;
  const bool want_mask_head = (flags & SM_TRACK_MASK_HEAD) != 0;
  Arena& search_arena = cur_->search;
  search_arena.reset();
  cur_->named.clear();
  Act xf = backbone(x, B, cfg_.search_size, search_arena, true, st);
  cur_->named["search"] = xf;
  const int nb = (want_feats || want_mask_head) ? 3 : 2;
  float* outs[3] = {cls, loc, mask};
  // all branches wanted: their conv_search layers run as ONE GEMM over xf (N = 256 x branches)
  const bool use_cat = nb == n_branches_ && cfg_.backend == SM_BACKEND_TENSOR;
  Act cs_all;
  if (use_cat) cs_all = conv(xf, L(kSearchCat), true, nullptr, search_arena, st);
  for (int br = 0; br < nb; ++br) {
    // the branches only share their input: run them side by side (their 1x1 heads and the xcorr do not fill
    // the GPU on their own)
    cudaStream_t bs = (concurrent() && br > 0) ? cur_->aux[br - 1] : st;
    order_after(st, bs);
    const std::string P = kBranch[br];
    Act cs = use_cat ? cs_all : conv(xf, L(P + "conv_search.0"), true, nullptr, search_arena, bs);
    Act corr = alloc_act(search_arena, B, cs.H - 4, cs.W - 4, 256);
    const size_t off = ((size_t)br * cfg_.num_slots + slot0) * 25 * 256;
    {
      Scope sc(this, std::string(kCorrName[br]), "xcorr", 2.0 * 25 * corr.numel(),
               4.0 * (2.0 * corr.numel() + (double)B * cs.H * cs.W * 256 + (double)B * 25 * 256), bs);
      corr.sexp = tscale(kCorrName[br]);
      const int s_kc = L(P + "conv_kernel.0").s_out;
      launch_xcorr_nhwc(cs, use_cat ? 256 * br : 0, kcache_hi_ + off, exact_ ? kcache_lo_ + off : nullptr, 5, 5, corr,
                        std::ldexp(1.f, corr.sexp - cs.sexp - s_kc), ovf_flag_, bs);
      ++launches_;
      last_end_[corr.hi] = +1;
    }
    note_tensor(corr, kCorrName[br], bs);
    cur_->named[kCorrName[br]] = corr;
    if (!(br == 2 && !want_mask_head)) {
      Act h = conv(corr, L(P + "head.0"), true, nullptr, search_arena, bs);
      Epilogue ep;
      ep.relu = 0;
      ep.out_mode = OUT_NCHW_F32;
      ep.out_f32 = outs[br];
      conv_into(h, L(P + "head.3"), ep, bs);
    }
  }
  for (int br = 1; br < nb; ++br) order_after((concurrent()) ? cur_->aux[br - 1] : st, st);
}

F32T Engine::small(const F32T& a, const F32T* b, int Ho, const ConvW& Lw, bool relu, float* out_override, Arena& ar,
                   cudaStream_t st) {
  F32T out;
  out.B = a.B; out.H = Ho; out.W = Ho; out.C = Lw.g.Cout;
  out.p = out_override != nullptr ? out_override
                                  : static_cast<float*>(ar.alloc((size_t)a.B * Ho * Ho * Lw.g.Cout * sizeof(float)));
  SMK_CHECK(a.C == Lw.g.Cin && (b == nullptr || (b->C == a.C && b->H == a.H)), "small conv operand shapes");
  const int* map = updown_map(Ho, a.H);
  Scope sc(this, Lw.conv_key, "refine_small", 2.0 * a.B * Ho * Ho * 9.0 * a.C * Lw.g.Cout,
           4.0 * a.B * ((double)a.H * a.W * a.C * (b ? 2 : 1) + (double)Ho * Ho * Lw.g.Cout), st);
  launch_small_conv3x3_maps(a.p, b ? b->p : nullptr, a.B, a.H, a.W, Ho, Ho, a.C, Lw.g.Cout, map, map, Lw.w_ref, Lw.beta,
                            relu ? 1 : 0, out.p, st);
  ++launches_;
  return out;
}

// Refine.forward(test=True), custom.py:131-154, one (dy,dx) per stream
void Engine::do_refine(int B, const int32_t* pos, float* out, cudaStream_t st) {
  SMK_CHECK(have_mask_feats_ && B == last_B_, "sm_refine must follow sm_track(..., SM_TRACK_MASK_FEATURES) with the same B");
  join_lanes(st);
  const std::vector<uint64_t> key = {2, (uint64_t)B, (uint64_t)pos, (uint64_t)out, (uint64_t)st,
                                     (uint64_t)lanes_[0].named["p0"].hi};
  run_with_graph(key, st, [&] { refine_impl(B, pos, out, st); });
}

void Engine::refine_impl(int B, const int32_t* pos, float* out, cudaStream_t st) {
  SMK_CHECK(cfg_.with_mask, "engine was built without the mask branch");
  SMK_CHECK(have_mask_feats_ && B == last_B_, "sm_refine must follow sm_track(..., SM_TRACK_MASK_FEATURES) with the same B");
  // same split as the track that cached the features
  LaneGuard guard{this, st};
  fork_lanes(st);
  for (int l = split_n_ - 1; l >= 0; --l) {
    cur_ = &lanes_[l];
    const int b0 = split_off_[l], nbat = split_off_[l + 1] - split_off_[l];
    cudaStream_t ls = (l == 0 || !concurrent()) ? st : lanes_[l].own;
    refine_lane(nbat, pos + 2 * b0, out + (size_t)b0 * 127 * 127, ls);
  }
  cur_ = &lanes_[0];
  guard.armed = false;
  join_forked(st);
}

void Engine::refine_lane(int B, const int32_t* pos, float* out, cudaStream_t st) {
  Arena& ar = cur_->refine;
  ar.reset();
  const std::string R = "refine_model.";
  const Act& p0 = cur_->named["p0"];
  const Act& p1 = cur_->named["p1"];
  const Act& p2 = cur_->named["p2"];
  const Act& corr = cur_->named["corr_mask"];
  // The three v-branches (crop -> conv -> conv on p2 / p1 / p0) depend only on the cached pyramid: they run on
  // auxiliary streams while the main stream walks deconv -> h2 -> post0 -> h1 -> post1 -> h0 -> post2.
  cudaStream_t s2 = concurrent() ? cur_->aux[0] : st, s1 = concurrent() ? cur_->aux[1] : st,
               s0 = concurrent() ? cur_->aux[2] : st;
  order_after(st, s2);
  order_after(st, s1);
  order_after(st, s0);
  // level 2 branch (15x15)
  Act c2 = alloc_act(ar, B, 15, 15, 512);
  {
    Scope sc(this, "crop_p2", "refine_misc", 0, 8.0 * c2.numel(), s2);
    last_end_[c2.hi] = +1;
    c2.sexp = p2.sexp;
    if (calibrating_) tensor_name_[c2.hi] = tensor_name_[p2.hi];
    launch_refine_crop(p2, pos, R_ - 1, 1, 4, 15, c2, s2); ++launches_;
  }
  Act v2a = conv(c2, L(R + "v2.0"), true, nullptr, ar, s2);
  F32T v2b = conv_f32(v2a, L(R + "v2.2"), true, ar, s2);
  // level 1 branch (31x31)
  Act c1 = alloc_act(ar, B, 31, 31, 256);
  {
    Scope sc(this, "crop_p1", "refine_misc", 0, 8.0 * c1.numel(), s1);
    last_end_[c1.hi] = +1;
    c1.sexp = p1.sexp;
    if (calibrating_) tensor_name_[c1.hi] = tensor_name_[p1.hi];
    launch_refine_crop(p1, pos, R_ - 1, 2, 8, 31, c1, s1); ++launches_;
  }
  Act v1a = conv(c1, L(R + "v1.0"), true, nullptr, ar, s1);
  F32T v1b = conv_f32(v1a, L(R + "v1.2"), true, ar, s1);
  // level 0 branch (61x61)
  Act c0 = alloc_act(ar, B, 61, 61, 64);
  {
    Scope sc(this, "crop_p0", "refine_misc", 0, 8.0 * c0.numel(), s0);
    last_end_[c0.hi] = +1;
    c0.sexp = p0.sexp;
    if (calibrating_) tensor_name_[c0.hi] = tensor_name_[p0.hi];
    launch_refine_crop(p0, pos, R_ - 1, 4, 16, 61, c0, s0); ++launches_;
  }
  F32T v0a = conv_f32(c0, L(R + "v0.0"), true, ar, s0);
  F32T v0b = small(v0a, nullptr, 61, L(R + "v0.2"), true, nullptr, ar, s0);
  // main chain: p3 = corr_feature[:, :, dy, dx]; out = deconv(p3)
  float* p3 = static_cast<float*>(ar.alloc((size_t)B * 256 * sizeof(float)));
  F32T d = alloc_f32(ar, B, 15, 15, 32);
  {
    Scope sc(this, "deconv", "refine_misc", 2.0 * B * 256 * 7200, 4.0 * (256.0 * 7200 + B * 7200.0), st);
    launch_gather_corr(corr, pos, p3, std::ldexp(1.f, -corr.sexp), st); ++launches_;
    launch_deconv(p3, deconv_w_, deconv_b_, d.p, B, 256, 7200, 32, st); ++launches_;
  }
  F32T h2a = small(d, nullptr, 15, L(R + "h2.0"), true, nullptr, ar, st);
  F32T h2b = small(h2a, nullptr, 15, L(R + "h2.2"), true, nullptr, ar, st);
  order_after(s2, st);
  F32T o0 = small(h2b, &v2b, 31, L(R + "post0"), false, nullptr, ar, st);   // post0(up31(h2 + v2))
  F32T h1a = small(o0, nullptr, 31, L(R + "h1.0"), true, nullptr, ar, st);
  F32T h1b = small(h1a, nullptr, 31, L(R + "h1.2"), true, nullptr, ar, st);
  order_after(s1, st);
  F32T o1 = small(h1b, &v1b, 61, L(R + "post1"), false, nullptr, ar, st);   // post1(up61(h1 + v1))
  F32T h0a = small(o1, nullptr, 61, L(R + "h0.0"), true, nullptr, ar, st);
  F32T h0b = small(h0a, nullptr, 61, L(R + "h0.2"), true, nullptr, ar, st);
  order_after(s0, st);
  small(h0b, &v0b, 127, L(R + "post2"), false, out, ar, st);                // (B,127,127,1) == (B,127*127)
}

// Host-buffer step, asynchronous: H2D on a copy stream, compute on the caller's stream, D2H on a second copy
// stream, chained by events.  Two staging sets alternate, so submitting step k+1 before waiting for step k overlaps
// its input transfer (and step k's result transfer) with compute.  Returns the ticket to pass to host_wait().
int Engine::track_host_async(int slot0, int B, const float* xh, float* clsh, float* loch, const int32_t* posh,
                             float* maskh, cudaStream_t st) {
  const size_t S = cfg_.search_size, A = cfg_.anchor_num;
  const size_t nx = (size_t)B * 3 * S * S, ncls = (size_t)B * 2 * A * R_ * R_, nloc = 2 * ncls;
  SMK_CHECK(B >= 1 && B <= cfg_.max_batch, "batch");
  const int t = (int)(host_calls_++ & 1);
  if (set_busy_[t]) host_wait(t);                 // the staging set is still owned by an un-waited ticket
  const bool refine = posh != nullptr && maskh != nullptr;
  SMK_CUDA(cudaMemcpyAsync(stage_x_[t], xh, nx * sizeof(float), cudaMemcpyHostToDevice, h2d_stream_));
  if (refine)
    SMK_CUDA(cudaMemcpyAsync(stage_pos_[t], posh, (size_t)B * 2 * sizeof(int32_t), cudaMemcpyHostToDevice, h2d_stream_));
  SMK_CUDA(cudaEventRecord(h2d_done_[t], h2d_stream_));
  if (lanes_for(n_lanes_, B) >= 2 && !use_graphs_ && concurrent()) {
    // decoupled lanes (see lanes_dirty_): order them after the caller's stream once (templates written there), then
    // each lane only depends on its inputs
    SMK_CHECK(weights_ready_, "weights not loaded");
    SMK_CHECK(slot0 >= 0 && slot0 + B <= cfg_.num_slots, "track batch/slot range");
    SMK_CHECK(!refine || cfg_.with_mask, "engine was built without the mask branch");
    split_batch(B);
    for (int l = split_n_ - 1; l >= 0; --l) {
      cur_ = &lanes_[l];
      cudaStream_t ls = cur_->own;
      const int b0 = split_off_[l], nbat = split_off_[l + 1] - split_off_[l];
      order_after(st, ls);
      SMK_CUDA(cudaStreamWaitEvent(ls, h2d_done_[t], 0));
      track_lane(slot0 + b0, nbat, stage_x_[t] + b0 * 3 * S * S, stage_cls_[t] + b0 * 2 * A * R_ * R_,
                 stage_loc_[t] + b0 * 4 * A * R_ * R_, nullptr, refine ? SM_TRACK_MASK_FEATURES : 0, ls);
      if (refine) refine_lane(nbat, stage_pos_[t] + 2 * b0, stage_mask_[t] + (size_t)b0 * 127 * 127, ls);
      SMK_CUDA(cudaEventRecord(lane_done_[t][l], ls));
      SMK_CUDA(cudaStreamWaitEvent(d2h_stream_, lane_done_[t][l], 0));
    }
    cur_ = &lanes_[0];
    last_B_ = B;
    have_mask_feats_ = refine;
    lanes_dirty_ = true;
  } else {
  SMK_CUDA(cudaStreamWaitEvent(st, h2d_done_[t], 0));
  // lane 1 stays forked between its track and its refine (nobody reads cls/loc on `st` in between)
  defer_join_ = refine && !use_graphs_;
  try {
    do_track(slot0, B, stage_x_[t], stage_cls_[t], stage_loc_[t], nullptr, refine ? SM_TRACK_MASK_FEATURES : 0, st);
  } catch (...) {
    defer_join_ = false;
    throw;
  }
  defer_join_ = false;
  if (refine) do_refine(B, stage_pos_[t], stage_mask_[t], st);
  SMK_CUDA(cudaEventRecord(compute_done_[t], st));
  SMK_CUDA(cudaStreamWaitEvent(d2h_stream_, compute_done_[t], 0));
  }
  SMK_CUDA(cudaMemcpyAsync(clsh, stage_cls_[t], ncls * sizeof(float), cudaMemcpyDeviceToHost, d2h_stream_));
  SMK_CUDA(cudaMemcpyAsync(loch, stage_loc_[t], nloc * sizeof(float), cudaMemcpyDeviceToHost, d2h_stream_));
  if (refine)
    SMK_CUDA(cudaMemcpyAsync(maskh, stage_mask_[t], (size_t)B * 127 * 127 * sizeof(float), cudaMemcpyDeviceToHost, d2h_stream_));
  SMK_CUDA(cudaEventRecord(d2h_done_[t], d2h_stream_));
  set_busy_[t] = true;
  return t;
}

void Engine::host_wait(int ticket) {
  SMK_CHECK(ticket == 0 || ticket == 1, "bad ticket");
  if (!set_busy_[ticket]) return;
  SMK_CUDA(cudaEventSynchronize(d2h_done_[ticket]));
  set_busy_[ticket] = false;
}

void Engine::track_host(int slot0, int B, const float* xh, float* clsh, float* loch, const int32_t* posh, float* maskh,
                        cudaStream_t st) {
  host_wait(track_host_async(slot0, B, xh, clsh, loch, posh, maskh, st));
}


// ------------------------------------------------------------------------------------------------
// Whole frame of siamese_track (tools/test.py:201-261) without leaving the device: track(_mask) -> score/box
// post-processing + argmax (:205-254) -> track_refine at the position that argmax selected (:253-257).  Each lane runs
// its share of the streams start to end on its own stream; the lanes only meet at the end of the call.
namespace {
Engine::StepIO slice_io(const Engine::StepIO& io, int b0, size_t S, size_t A, size_t RR) {
  Engine::StepIO o = io;
  o.x = io.x + (size_t)b0 * 3 * S * S;
  o.tsz = io.tsz + 2 * (size_t)b0;
  o.cls = io.cls + (size_t)b0 * 2 * A * RR;
  o.loc = io.loc + (size_t)b0 * 4 * A * RR;
  if (io.mask) o.mask = io.mask + (size_t)b0 * 3969 * RR;
  o.best = io.best + b0;
  o.pos = io.pos + 2 * (size_t)b0;
  o.rec = io.rec + 8 * (size_t)b0;
  if (io.refine) o.refine = io.refine + (size_t)b0 * 127 * 127;
  if (io.mask_col) o.mask_col = io.mask_col + (size_t)b0 * 3969;
  return o;
}
}  // namespace

void Engine::step_lane(int slot0, int B, const StepIO& io, cudaStream_t st) {
  track_lane(slot0, B, io.x, io.cls, io.loc, io.mask, io.flags, st);
  {
    Scope sc(this, "select", "select", 0, 4.0 * B * 6.0 * cfg_.anchor_num * R_ * R_, st);
    launch_select(io.cls, io.loc, io.anchors, io.window, io.tsz, B, cfg_.anchor_num, R_, io.penalty_k,
                  io.window_influence, io.best, io.pos, io.rec, st);
    ++launches_;
  }
  if (io.refine != nullptr) refine_lane(B, io.pos, io.refine, st);
  if (io.mask_col != nullptr) {
    launch_gather_mask_col(io.mask, io.pos, B, 3969, R_, io.mask_col, st);
    ++launches_;
  }
}

void Engine::do_step(int slot0, int B, const StepIO& io, cudaStream_t st) {
  SMK_CHECK(weights_ready_, "weights not loaded");
  SMK_CHECK(B >= 1 && B <= cfg_.max_batch && slot0 >= 0 && slot0 + B <= cfg_.num_slots, "step batch/slot range");
  SMK_CHECK(io.x && io.tsz && io.anchors && io.window && io.cls && io.loc && io.best && io.pos && io.rec, "null argument");
  const bool want_feats = (io.flags & SM_TRACK_MASK_FEATURES) != 0, want_head = (io.flags & SM_TRACK_MASK_HEAD) != 0;
  SMK_CHECK(!(want_feats || want_head || io.refine) || cfg_.with_mask, "engine was built without the mask branch");
  SMK_CHECK(io.refine == nullptr || want_feats, "refine output needs SM_TRACK_MASK_FEATURES");
  SMK_CHECK(!want_head || io.mask != nullptr, "mask output buffer required");
  SMK_CHECK(io.mask_col == nullptr || want_head, "mask column needs SM_TRACK_MASK_HEAD");
  join_lanes(st);
  const std::vector<uint64_t> key = {3, (uint64_t)slot0, (uint64_t)B, (uint64_t)io.x, (uint64_t)io.tsz, (uint64_t)io.cls,
                                     (uint64_t)io.loc, (uint64_t)io.mask, (uint64_t)io.flags, (uint64_t)io.pos,
                                     (uint64_t)io.rec, (uint64_t)io.refine, (uint64_t)io.mask_col, (uint64_t)st,
                                     (uint64_t)io.anchors, (uint64_t)io.window};
  run_with_graph(key, st, [&] {
    split_batch(B);
    LaneGuard guard{this, st};
    const size_t S = cfg_.search_size, A = cfg_.anchor_num, RR = (size_t)R_ * R_;
    fork_lanes(st);
    for (int l = split_n_ - 1; l >= 0; --l) {
      cur_ = &lanes_[l];
      const int b0 = split_off_[l], nbat = split_off_[l + 1] - split_off_[l];
      cudaStream_t ls = (l == 0 || !concurrent()) ? st : lanes_[l].own;
      step_lane(slot0 + b0, nbat, slice_io(io, b0, S, A, RR), ls);
    }
    cur_ = &lanes_[0];
    guard.armed = false;
    join_forked(st);
    last_B_ = B;
    have_mask_feats_ = want_feats || want_head;
  });
}

// Host-buffer form of do_step (pinned buffers recommended): H2D of the frames and of target_sz*scale_x, the whole
// frame on the device, D2H of the per-stream records (+ refine logits / mask column / cls / loc when asked for).
// Same ticket / staging-set protocol as track_host_async.
int Engine::step_host_async(int slot0, int B, const sm_step_io& h, cudaStream_t st) {
  const size_t S = cfg_.search_size, A = cfg_.anchor_num, RR = (size_t)R_ * R_;
  SMK_CHECK(B >= 1 && B <= cfg_.max_batch, "batch");
  SMK_CHECK(weights_ready_, "weights not loaded");
  SMK_CHECK(slot0 >= 0 && slot0 + B <= cfg_.num_slots, "step batch/slot range");
  SMK_CHECK(h.x_host && h.tsz_host && h.anchors_dev && h.window_dev && h.records_host, "null argument");
  const bool want_feats = (h.flags & SM_TRACK_MASK_FEATURES) != 0, want_head = (h.flags & SM_TRACK_MASK_HEAD) != 0;
  SMK_CHECK(!(want_feats || want_head || h.refine_host) || cfg_.with_mask, "engine was built without the mask branch");
  SMK_CHECK(h.refine_host == nullptr || want_feats, "refine output needs SM_TRACK_MASK_FEATURES");
  SMK_CHECK(h.mask_col_host == nullptr || want_head, "mask column needs SM_TRACK_MASK_HEAD");
  if (want_head && mask_raw_ == nullptr)
    SMK_CUDA(cudaMalloc(&mask_raw_, (size_t)cfg_.max_batch * 3969 * RR * sizeof(float)));
  const int t = (int)(host_calls_++ & 1);
  if (set_busy_[t]) host_wait(t);
  SMK_CUDA(cudaMemcpyAsync(stage_x_[t], h.x_host, (size_t)B * 3 * S * S * sizeof(float), cudaMemcpyHostToDevice, h2d_stream_));
  SMK_CUDA(cudaMemcpyAsync(stage_tsz_[t], h.tsz_host, (size_t)B * 2 * sizeof(double), cudaMemcpyHostToDevice, h2d_stream_));
  SMK_CUDA(cudaEventRecord(h2d_done_[t], h2d_stream_));
  StepIO io;
  io.x = stage_x_[t]; io.tsz = stage_tsz_[t]; io.anchors = h.anchors_dev; io.window = h.window_dev;
  io.penalty_k = h.penalty_k; io.window_influence = h.window_influence; io.flags = h.flags;
  io.cls = stage_cls_[t]; io.loc = stage_loc_[t]; io.mask = want_head ? mask_raw_ : nullptr;
  io.best = stage_best_[t]; io.pos = stage_pos_[t]; io.rec = stage_rec_[t];
  io.refine = h.refine_host != nullptr ? stage_mask_[t] : nullptr;
  io.mask_col = h.mask_col_host != nullptr ? stage_maskcol_[t] : nullptr;
  if (lanes_for(n_lanes_, B) >= 2 && !use_graphs_ && concurrent()) {
    split_batch(B);
    for (int l = split_n_ - 1; l >= 0; --l) {
      cur_ = &lanes_[l];
      cudaStream_t ls = cur_->own;
      const int b0 = split_off_[l], nbat = split_off_[l + 1] - split_off_[l];
      order_after(st, ls);
      SMK_CUDA(cudaStreamWaitEvent(ls, h2d_done_[t], 0));
      step_lane(slot0 + b0, nbat, slice_io(io, b0, S, A, RR), ls);
      SMK_CUDA(cudaEventRecord(lane_done_[t][l], ls));
      SMK_CUDA(cudaStreamWaitEvent(d2h_stream_, lane_done_[t][l], 0));
    }
    cur_ = &lanes_[0];
    last_B_ = B;
    have_mask_feats_ = want_feats || want_head;
    lanes_dirty_ = true;
  } else {
    SMK_CUDA(cudaStreamWaitEvent(st, h2d_done_[t], 0));
    do_step(slot0, B, io, st);
    SMK_CUDA(cudaEventRecord(compute_done_[t], st));
    SMK_CUDA(cudaStreamWaitEvent(d2h_stream_, compute_done_[t], 0));
  }
  SMK_CUDA(cudaMemcpyAsync(h.records_host, stage_rec_[t], (size_t)B * 8 * sizeof(float), cudaMemcpyDeviceToHost, d2h_stream_));
  if (h.refine_host)
    SMK_CUDA(cudaMemcpyAsync(h.refine_host, stage_mask_[t], (size_t)B * 127 * 127 * sizeof(float), cudaMemcpyDeviceToHost, d2h_stream_));
  if (h.mask_col_host)
    SMK_CUDA(cudaMemcpyAsync(h.mask_col_host, stage_maskcol_[t], (size_t)B * 3969 * sizeof(float), cudaMemcpyDeviceToHost, d2h_stream_));
  if (h.cls_host)
    SMK_CUDA(cudaMemcpyAsync(h.cls_host, stage_cls_[t], (size_t)B * 2 * A * RR * sizeof(float), cudaMemcpyDeviceToHost, d2h_stream_));
  if (h.loc_host)
    SMK_CUDA(cudaMemcpyAsync(h.loc_host, stage_loc_[t], (size_t)B * 4 * A * RR * sizeof(float), cudaMemcpyDeviceToHost, d2h_stream_));
  SMK_CUDA(cudaEventRecord(d2h_done_[t], d2h_stream_));
  set_busy_[t] = true;
  return t;
}

void Engine::do_export(const char* what, float* out, int64_t* shape4, cudaStream_t st) {
  join_lanes(st);
  if (std::string(what) == "zf") {
    SMK_CHECK(have_zf_, "no cached tensor named 'zf'");
    if (shape4 != nullptr) { shape4[0] = zf_.B; shape4[1] = zf_.C; shape4[2] = zf_.H; shape4[3] = zf_.W; }
    if (out != nullptr) { launch_split_to_f32(zf_, out, st, std::ldexp(1.f, -zf_.sexp)); ++launches_; }
    return;
  }
  int total_B = 0;
  for (int l = 0; l < split_n_; ++l) {       // the lanes hold consecutive blocks of streams
    auto it = lanes_[l].named.find(what);
    SMK_CHECK(it != lanes_[l].named.end(), std::string("no cached tensor named '") + what + "'");
    const Act& a = it->second;
    if (shape4 != nullptr) { shape4[1] = a.C; shape4[2] = a.H; shape4[3] = a.W; }
    if (out != nullptr) {
      launch_split_to_f32(a, out + (size_t)total_B * a.C * a.H * a.W, st, std::ldexp(1.f, -a.sexp));
      ++launches_;
    }
    total_B += a.B;
  }
  if (shape4 != nullptr) shape4[0] = total_B;
}

std::string Engine::profile_dump() {
  SMK_CUDA(cudaDeviceSynchronize());
  std::string out;
  for (auto& r : prof_) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, r.e0, r.e1);
    char line[512];
    snprintf(line, sizeof line, "%s\t%s\t%.6f\t%.0f\t%.0f\n", r.name.c_str(), r.cat.c_str(), ms, r.flops, r.bytes);
    out += line;
    event_pool_.push_back(r.e0);
    event_pool_.push_back(r.e1);
  }
  prof_.clear();
  return out;
}

// ================================================================================================
// standalone conv operator (kernel-level parity tests)

static void conv2d_op(const float* x, const float* w, const float* scale, const float* shift, float* out, int B,
                      int Cin, int H, int W, int Cout, int KH, int KW, int stride, int pad, int dil, int relu,
                      int backend, int precision, cudaStream_t st) {
  ConvGeom g{Cin, Cout, KH, KW, stride, pad, dil};
  const bool exact = precision == SM_PRECISION_EXACT;
  const bool use_gemm = backend == SM_BACKEND_TENSOR;
  SMK_CHECK(!use_gemm || gemm_conv_supported(g), "tensor-core conv needs Cin % 64 == 0");
  const size_t K = (size_t)KH * KW * Cin;
  const int cout_pad = use_gemm ? gemm_cout_pad(Cout) : Cout;
  std::vector<float> hw(K * Cout), hs(Cout, 1.f), hb(Cout, 0.f);
  SMK_CUDA(cudaStreamSynchronize(st));
  SMK_CUDA(cudaMemcpy(hw.data(), w, hw.size() * sizeof(float), cudaMemcpyDeviceToHost));
  if (scale) SMK_CUDA(cudaMemcpy(hs.data(), scale, Cout * sizeof(float), cudaMemcpyDeviceToHost));
  if (shift) SMK_CUDA(cudaMemcpy(hb.data(), shift, Cout * sizeof(float), cudaMemcpyDeviceToHost));
  std::vector<float> wref(K * Cout), alpha(cout_pad, 0.f), beta(cout_pad, 0.f);
  std::vector<__half> whi((size_t)cout_pad * K, __float2half_rn(0.f)), wlo((size_t)cout_pad * K, __float2half_rn(0.f));
  const int HW = KH * KW;
  for (int n = 0; n < Cout; ++n) {
    float amax = 0.f;
    for (int c = 0; c < Cin; ++c)
      for (int t = 0; t < HW; ++t) {
        const float fw = (float)((double)hw[((size_t)n * Cin + c) * HW + t] * (double)hs[n]);
        wref[((size_t)t * Cin + c) * Cout + n] = fw;
        amax = std::max(amax, std::fabs(fw));
      }
    beta[n] = hb[n];
    alpha[n] = 1.f;
    if (use_gemm) {
      int e = amax > 0.f ? (int)std::floor(std::log2(16384.0 / (double)amax)) : 0;
      e = std::max(-24, std::min(24, e));
      alpha[n] = std::ldexp(1.f, -e);
      for (int c = 0; c < Cin; ++c)
        for (int t = 0; t < HW; ++t) {
          const float fw = std::ldexp(wref[((size_t)t * Cin + c) * Cout + n], e);
          const __half h = __float2half_rn(fw);
          whi[((size_t)n * HW + t) * Cin + c] = h;
          wlo[((size_t)n * HW + t) * Cin + c] = __float2half_rn(fw - __half2float(h));
        }
    }
  }
  const int Ho = g.out_size(H), Wo = g.out_size(W);
  Act in;
  in.B = B; in.H = H; in.W = W; in.C = Cin;
  __half *d_whi = nullptr, *d_wlo = nullptr;
  float *d_wref = nullptr, *d_alpha = nullptr, *d_beta = nullptr;
  SMK_CUDA(cudaMalloc(&in.hi, in.numel() * sizeof(__half)));
  if (exact) SMK_CUDA(cudaMalloc(&in.lo, in.numel() * sizeof(__half)));
  SMK_CUDA(cudaMalloc(&d_whi, whi.size() * sizeof(__half)));
  SMK_CUDA(cudaMalloc(&d_wlo, wlo.size() * sizeof(__half)));
  SMK_CUDA(cudaMalloc(&d_wref, wref.size() * sizeof(float)));
  SMK_CUDA(cudaMalloc(&d_alpha, alpha.size() * sizeof(float)));
  SMK_CUDA(cudaMalloc(&d_beta, beta.size() * sizeof(float)));
  SMK_CUDA(cudaMemcpy(d_whi, whi.data(), whi.size() * sizeof(__half), cudaMemcpyHostToDevice));
  SMK_CUDA(cudaMemcpy(d_wlo, wlo.data(), wlo.size() * sizeof(__half), cudaMemcpyHostToDevice));
  SMK_CUDA(cudaMemcpy(d_wref, wref.data(), wref.size() * sizeof(float), cudaMemcpyHostToDevice));
  SMK_CUDA(cudaMemcpy(d_alpha, alpha.data(), alpha.size() * sizeof(float), cudaMemcpyHostToDevice));
  SMK_CUDA(cudaMemcpy(d_beta, beta.data(), beta.size() * sizeof(float), cudaMemcpyHostToDevice));
  launch_import_nchw(x, in, st);
  Epilogue ep;
  ep.alpha = d_alpha;
  ep.beta = d_beta;
  ep.relu = relu;
  ep.out_mode = OUT_NCHW_F32;
  ep.out_f32 = out;
  int dev = 0, sms = 148;
  SMK_CUDA(cudaGetDevice(&dev));
  SMK_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  (void)Ho; (void)Wo;
  if (use_gemm && patch_conv_supported(in, g)) {
    // the engine runs this geometry on the resident-patch kernel (NHWC split output): same here, then export
    Act o;
    o.B = B; o.H = Ho; o.W = Wo; o.C = Cout;
    SMK_CUDA(cudaMalloc(&o.hi, o.numel() * sizeof(__half)));
    if (exact) SMK_CUDA(cudaMalloc(&o.lo, o.numel() * sizeof(__half)));
    Epilogue e2 = ep;
    e2.out_mode = OUT_NHWC_SPLIT;
    e2.out_hi = o.hi;
    e2.out_lo = o.lo;
    e2.out_f32 = nullptr;
    launch_conv3x3_patch(in, g, d_whi, d_wlo, (int)K, e2, exact ? 2 : 1, sms, st);
    launch_split_to_f32(o, out, st);
    SMK_CUDA(cudaStreamSynchronize(st));
    cudaFree(o.hi); cudaFree(o.lo);
  } else if (use_gemm) launch_gemm_conv(in, g, d_whi, d_wlo, cout_pad, ep, exact ? 2 : 1, sms, st);
  else launch_ref_conv(in, g, d_wref, ep, st);
  SMK_CUDA(cudaStreamSynchronize(st));
  cudaFree(in.hi); cudaFree(in.lo); cudaFree(d_whi); cudaFree(d_wlo); cudaFree(d_wref); cudaFree(d_alpha); cudaFree(d_beta);
}

}  // namespace smk

// ================================================================================================
// C ABI

struct sm_engine {
  std::unique_ptr<smk::Engine> impl;
};

#define SM_API_BEGIN try {
#define SM_API_END                                  \
  return 0;                                         \
  }                                                 \
  catch (const std::exception& ex) {                \
    smk::g_last_error = ex.what();                  \
    return -1;                                      \
  }                                                 \
  catch (...) {                                     \
    smk::g_last_error = "unknown error";            \
    return -1;                                      \
  }

extern "C" {

const char* sm_last_error(void) { return smk::g_last_error.c_str(); }
const char* sm_version(void) { return "siammask_b200 0.1 (sm_100a)"; }

int sm_engine_create(const sm_config* cfg, sm_engine** out) {
  SM_API_BEGIN
  SMK_CHECK(cfg != nullptr && out != nullptr, "null argument");
  int ndev = 0;
  cudaError_t err = cudaGetDeviceCount(&ndev);
  SMK_CHECK(err == cudaSuccess && ndev > 0, "no CUDA device: siammask_b200 has no CPU fallback");
  auto* e = new sm_engine;
  try {
    e->impl.reset(new smk::Engine(*cfg));
  } catch (...) {
    delete e;
    throw;
  }
  *out = e;
  SM_API_END
}

void sm_engine_destroy(sm_engine* e) { delete e; }

int sm_engine_load_weights(sm_engine* e, const sm_tensor_desc* tensors, int32_t n) {
  SM_API_BEGIN
  SMK_CHECK(e && tensors && n > 0, "null argument");
  e->impl->load_weights(tensors, n);
  SM_API_END
}

int sm_engine_weight_blob(sm_engine* e, void** dev_ptr, size_t* bytes) {
  SM_API_BEGIN
  SMK_CHECK(e && dev_ptr && bytes, "null argument");
  e->impl->weight_blob(dev_ptr, bytes);
  SM_API_END
}

int sm_engine_adopt_weights(sm_engine* e) {
  SM_API_BEGIN
  SMK_CHECK(e, "null argument");
  e->impl->adopt_weights();
  SM_API_END
}

int sm_engine_calibrate(sm_engine* e, int32_t B, const float* z_nchw, const float* x_nchw, void* stream) {
  SM_API_BEGIN
  SMK_CHECK(e && z_nchw && x_nchw, "null argument");
  e->impl->calibrate(B, z_nchw, x_nchw, static_cast<cudaStream_t>(stream));
  SM_API_END
}

int sm_engine_status(sm_engine* e, int32_t* flags) {
  SM_API_BEGIN
  SMK_CHECK(e && flags, "null argument");
  *flags = e->impl->status();
  SM_API_END
}

int sm_template(sm_engine* e, int32_t slot0, int32_t B, const float* z, void* stream) {
  SM_API_BEGIN
  SMK_CHECK(e && z, "null argument");
  e->impl->do_template(slot0, B, z, static_cast<cudaStream_t>(stream));
  SM_API_END
}

int sm_track(sm_engine* e, int32_t slot0, int32_t B, const float* x, float* cls, float* loc, float* mask, int32_t flags,
             void* stream) {
  SM_API_BEGIN
  SMK_CHECK(e && x, "null argument");
  e->impl->do_track(slot0, B, x, cls, loc, mask, flags, static_cast<cudaStream_t>(stream));
  SM_API_END
}

int sm_refine(sm_engine* e, int32_t B, const int32_t* pos, float* out, void* stream) {
  SM_API_BEGIN
  SMK_CHECK(e && pos && out, "null argument");
  e->impl->do_refine(B, pos, out, static_cast<cudaStream_t>(stream));
  SM_API_END
}

int sm_track_host(sm_engine* e, int32_t slot0, int32_t B, const float* x_host, float* cls_host, float* loc_host,
                  const int32_t* pos_host, float* mask_out_host, void* stream) {
  SM_API_BEGIN
  SMK_CHECK(e && x_host && cls_host && loc_host, "null argument");
  e->impl->track_host(slot0, B, x_host, cls_host, loc_host, pos_host, mask_out_host, static_cast<cudaStream_t>(stream));
  SM_API_END
}

int sm_track_host_async(sm_engine* e, int32_t slot0, int32_t B, const float* x_host, float* cls_host, float* loc_host,
                        const int32_t* pos_host, float* mask_out_host, void* stream, int32_t* ticket) {
  SM_API_BEGIN
  SMK_CHECK(e && x_host && cls_host && loc_host && ticket, "null argument");
  *ticket = e->impl->track_host_async(slot0, B, x_host, cls_host, loc_host, pos_host, mask_out_host,
                                      static_cast<cudaStream_t>(stream));
  SM_API_END
}

int sm_track_host_wait(sm_engine* e, int32_t ticket) {
  SM_API_BEGIN
  SMK_CHECK(e, "null argument");
  e->impl->host_wait(ticket);
  SM_API_END
}

int sm_step(sm_engine* e, int32_t slot0, int32_t B, const float* x, const double* target_sz_in_crop, const float* anchors,
            const float* window, double penalty_k, double window_influence, int32_t flags, float* cls, float* loc,
            float* mask, int32_t* best_idx, int32_t* pos, float* records, float* refine_out, float* mask_col,
            void* stream) {
  SM_API_BEGIN
  SMK_CHECK(e, "null argument");
  smk::Engine::StepIO io;
  io.x = x; io.tsz = target_sz_in_crop; io.anchors = anchors; io.window = window;
  io.penalty_k = penalty_k; io.window_influence = window_influence; io.flags = flags;
  io.cls = cls; io.loc = loc; io.mask = mask; io.best = best_idx; io.pos = pos; io.rec = records;
  io.refine = refine_out; io.mask_col = mask_col;
  e->impl->do_step(slot0, B, io, static_cast<cudaStream_t>(stream));
  SM_API_END
}

int sm_step_host_async(sm_engine* e, int32_t slot0, int32_t B, const sm_step_io* io, void* stream, int32_t* ticket) {
  SM_API_BEGIN
  SMK_CHECK(e && io && ticket, "null argument");
  *ticket = e->impl->step_host_async(slot0, B, *io, static_cast<cudaStream_t>(stream));
  SM_API_END
}

int sm_xcorr_depthwise(const float* x, const float* k, float* out, int32_t B, int32_t C, int32_t H, int32_t W, int32_t kh,
                       int32_t kw, void* stream) {
  SM_API_BEGIN
  SMK_CHECK(x && k && out, "null argument");
  int ndev = 0;
  SMK_CHECK(cudaGetDeviceCount(&ndev) == cudaSuccess && ndev > 0, "no CUDA device: siammask_b200 has no CPU fallback");
  smk::launch_xcorr_nchw_f32(x, k, out, B * C, H, W, kh, kw, static_cast<cudaStream_t>(stream));
  SM_API_END
}

int sm_conv2d(const float* x, const float* w, const float* scale, const float* shift, float* out, int32_t B, int32_t Cin,
              int32_t H, int32_t W, int32_t Cout, int32_t KH, int32_t KW, int32_t stride, int32_t pad, int32_t dil,
              int32_t relu, int32_t backend, int32_t precision, void* stream) {
  SM_API_BEGIN
  SMK_CHECK(x && w && out, "null argument");
  int ndev = 0;
  SMK_CHECK(cudaGetDeviceCount(&ndev) == cudaSuccess && ndev > 0, "no CUDA device: siammask_b200 has no CPU fallback");
  smk::conv2d_op(x, w, scale, shift, out, B, Cin, H, W, Cout, KH, KW, stride, pad, dil, relu, backend, precision,
                 static_cast<cudaStream_t>(stream));
  SM_API_END
}

int sm_crop_resize(const uint8_t* frames, size_t frame_stride, int32_t H, int32_t W, const int32_t* boxes, int32_t B,
                   int32_t model_size, float* out, void* stream) {
  SM_API_BEGIN
  SMK_CHECK(frames && boxes && out && B >= 1 && H > 0 && W > 0 && model_size > 0, "bad argument");
  int ndev = 0;
  SMK_CHECK(cudaGetDeviceCount(&ndev) == cudaSuccess && ndev > 0, "no CUDA device: siammask_b200 has no CPU fallback");
  smk::launch_crop_resize(frames, frame_stride, H, W, boxes, B, model_size, out, static_cast<cudaStream_t>(stream));
  SM_API_END
}

int sm_warp_affine(const float* src, int32_t src_h, int32_t src_w, const double* maps, float* dst, int32_t dst_h,
                   int32_t dst_w, float border_value, int32_t B, void* stream) {
  SM_API_BEGIN
  SMK_CHECK(src && maps && dst && B >= 1 && src_h > 0 && src_w > 0 && dst_h > 0 && dst_w > 0, "bad argument");
  int ndev = 0;
  SMK_CHECK(cudaGetDeviceCount(&ndev) == cudaSuccess && ndev > 0, "no CUDA device: siammask_b200 has no CPU fallback");
  smk::launch_warp_affine(src, src_h, src_w, maps, dst, dst_h, dst_w, border_value, B, static_cast<cudaStream_t>(stream));
  SM_API_END
}

static smk::TrackerHp to_hp(const sm_tracker_hp* h) {
  smk::TrackerHp t;
  t.context_amount = h->context_amount; t.penalty_k = h->penalty_k; t.window_influence = h->window_influence; t.lr = h->lr;
  t.exemplar_size = h->exemplar_size; t.instance_size = h->instance_size; t.total_stride = h->total_stride;
  t.base_size = h->base_size; t.out_size = h->out_size; t.reserved = 0;
  return t;
}

int sm_tracker_prepare(int32_t B, const double* state, const int32_t* avg_chans, const sm_tracker_hp* hp, int32_t* boxes,
                       double* target_sz_in_crop, double* aux, void* stream) {
  SM_API_BEGIN
  SMK_CHECK(state && avg_chans && hp && boxes && target_sz_in_crop && aux && B >= 1, "bad argument");
  int ndev = 0;
  SMK_CHECK(cudaGetDeviceCount(&ndev) == cudaSuccess && ndev > 0, "no CUDA device: siammask_b200 has no CPU fallback");
  smk::launch_tracker_prepare(B, state, avg_chans, to_hp(hp), boxes, target_sz_in_crop, aux, static_cast<cudaStream_t>(stream));
  SM_API_END
}

int sm_tracker_update(int32_t B, double* state, const float* records, const double* aux, const int32_t* im_wh,
                      const sm_tracker_hp* hp, int32_t anchor_num, int32_t score_size, double* maps, double* out,
                      void* stream) {
  SM_API_BEGIN
  SMK_CHECK(state && records && aux && im_wh && hp && B >= 1 && score_size >= 1, "bad argument");
  int ndev = 0;
  SMK_CHECK(cudaGetDeviceCount(&ndev) == cudaSuccess && ndev > 0, "no CUDA device: siammask_b200 has no CPU fallback");
  smk::launch_tracker_update(B, state, records, aux, im_wh, to_hp(hp), anchor_num, score_size, maps, out,
                             static_cast<cudaStream_t>(stream));
  SM_API_END
}

int sm_select(sm_engine* e, int32_t B, const float* cls, const float* loc, const float* anchors, const float* window,
              const double* target_sz_in_crop, double penalty_k, double window_influence, int32_t* best_idx, int32_t* pos,
              float* records, void* stream) {
  SM_API_BEGIN
  SMK_CHECK(e && cls && loc && anchors && window && target_sz_in_crop && best_idx && pos && records, "null argument");
  SMK_CHECK(B >= 1, "batch");
  const sm_config& c = e->impl->cfg();
  const int R = (c.search_size - 127) / 8 + 9;
  smk::launch_select(cls, loc, anchors, window, target_sz_in_crop, B, c.anchor_num, R, penalty_k, window_influence,
                     best_idx, pos, records, static_cast<cudaStream_t>(stream));
  SM_API_END
}

int sm_export(sm_engine* e, const char* what, float* out, int64_t* shape4, void* stream) {
  SM_API_BEGIN
  SMK_CHECK(e && what, "null argument");
  e->impl->do_export(what, out, shape4, static_cast<cudaStream_t>(stream));
  SM_API_END
}

int sm_engine_set_graphs(sm_engine* e, int32_t on) {
  SM_API_BEGIN
  SMK_CHECK(e, "null argument");
  e->impl->set_graphs(on != 0);
  SM_API_END
}

int sm_profile_enable(sm_engine* e, int32_t on) {
  SM_API_BEGIN
  SMK_CHECK(e, "null argument");
  e->impl->set_profiling(on != 0);
  SM_API_END
}

int64_t sm_profile_dump(sm_engine* e, char* buf, size_t cap) {
  try {
    if (!e) return -1;
    static thread_local std::string pending;
    if (pending.empty()) pending = e->impl->profile_dump();
    if (buf == nullptr || cap <= pending.size()) return (int64_t)pending.size() + 1;
    std::memcpy(buf, pending.c_str(), pending.size() + 1);
    const int64_t n = (int64_t)pending.size();
    pending.clear();
    return n;
  } catch (const std::exception& ex) {
    smk::g_last_error = ex.what();
    return -1;
  }
}

int64_t sm_launch_count(const sm_engine* e) { return e ? e->impl->launches() : 0; }
size_t sm_engine_bytes(const sm_engine* e) { return e ? e->impl->bytes() : 0; }

}  // extern "C"
