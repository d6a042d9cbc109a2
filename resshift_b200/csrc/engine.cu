// Engine: the Swin-UNet denoiser of ResShift as a static program of sm_100a kernel launches, plus the
// residual-shift sampling loop, behind the C ABI declared in include/resshift_b200.h.
//
// Topology restates UNetModelSwin.__init__/forward (reference models/unet.py:659-895), ResBlock
// (:110-206), BasicLayer / SwinTransformerBlock (models/swin_transformer.py:163-281,348-442).
// Design notes (DESIGN.md has the long form):
//   * activations NHWC fp16; skip connections are written straight into the channel slice of the
//     decoder's concat buffer (th.cat at unet.py:891 costs nothing);
//   * every tensor lives in one caller-owned workspace; lifetimes are resolved at plan time;
//   * timestep embeddings (time_embed + all 22 emb_layers) are one small table computed by two tiny
//     kernels; in the sampling loop the table for all T steps is computed once.
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "../../include/resshift_b200.h"
#include "launch.cuh"
#include "vq_kernels.cuh"

namespace rs {

static thread_local std::string g_last_error;
void set_error(const std::string& msg) { g_last_error = msg; }
int fail(int code, const std::string& msg) { g_last_error = msg; return code; }

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

enum Role { R_CONV3 = 0, R_CONV1, R_LINEAR, R_BIAS, R_GN_W, R_GN_B, R_RELPOS, R_BUF_RELIDX, R_BUF_MASK, R_F32 /* fp32 tensor kept as is (VQ codebook) */ };

struct Param {
  std::string name;
  std::vector<int> shape;
  int role;
  size_t off = 0;        // byte offset in the arena
  size_t bytes = 0;
  int ipad = 0;          // padded input channels for weights
};

}  // namespace rs

using namespace rs;

struct rs_engine {
  int kind = 0;                 // 0: UNetModelSwin denoiser, 1: VQ-GAN first stage (vq.inc); the parameter store is shared
  rs_vq_config vq{};
  rs_unet_config cfg;
  std::vector<Param> params;
  std::map<std::string, int> index;
  size_t arena_bytes = 0;
  uint8_t* arena = nullptr;
  unsigned long long weights_epoch = 0;     // bumped by every rs_unet_load_param: tables derived from weights (FiLM) go stale
  // concatenated emb_layers ("FiLM") matrix: rows = sum 2*Cout over ResBlocks, K = time_embed_dim
  size_t film_w_off = 0, film_b_off = 0;
  int film_rows = 0;
  std::map<std::string, int> film_row_of;   // resblock prefix -> first row

  int time_dim() const { return cfg.model_channels * 4; }
  int fe_stages() const {
    if (cfg.lq_size == cfg.image_size) return 0;
    int s = 0, r = cfg.lq_size / cfg.image_size;
    while (r > 1) { r >>= 1; ++s; }
    return s;
  }
  int lq_in_ch() const { return cfg.cond_mask ? 4 : 3; }
  int lq_feat_ch() const { return fe_stages() == 0 ? lq_in_ch() : 16 << fe_stages(); }
  bool has_attn(int ds) const {
    for (int i = 0; i < cfg.n_attn; ++i) if (cfg.attention_resolutions[i] == ds) return true;
    return false;
  }
  const Param* find(const std::string& n) const {
    auto it = index.find(n);
    return it == index.end() ? nullptr : &params[it->second];
  }
  template <typename T> T* at(const std::string& n) const {
    const Param* p = find(n);
    return p ? reinterpret_cast<T*>(arena + p->off) : nullptr;
  }
};

// ------------------------------------------------------------------------------------------------
// architecture walk shared by the parameter inventory and the plan builder
// ------------------------------------------------------------------------------------------------
namespace {

struct Layer { int kind; int a, b; };   // kind: 0 conv(cin,cout) 1 res(cin,cout) 2 swin(c,res) 3 down(c) 4 up(c)
struct Topology {
  std::vector<std::vector<Layer>> input_blocks, output_blocks;
  std::vector<Layer> middle;
  std::vector<int> in_block_ch;    // output channels of each input block (the skip stack)
};

Topology build_topology(const rs_engine& e) {
  const rs_unet_config& c = e.cfg;
  Topology t;
  const int mc = c.model_channels;
  int ch = c.channel_mult[0] * mc;
  t.input_blocks.push_back({{0, c.in_channels + e.lq_feat_ch(), ch}});
  std::vector<int> chans{ch};
  int ds = c.image_size;
  for (int level = 0; level < c.n_levels; ++level) {
    for (int jj = 0; jj < c.num_res_blocks[level]; ++jj) {
      std::vector<Layer> layers{{1, ch, c.channel_mult[level] * mc}};
      ch = c.channel_mult[level] * mc;
      if (e.has_attn(ds) && jj == 0) layers.push_back({2, ch, ds});
      t.input_blocks.push_back(layers);
      chans.push_back(ch);
    }
    if (level != c.n_levels - 1) {
      t.input_blocks.push_back({{3, ch, ch}});
      chans.push_back(ch);
      ds /= 2;
    }
  }
  t.in_block_ch = chans;
  t.middle = {{1, ch, ch}, {2, ch, ds}, {1, ch, ch}};
  for (int level = c.n_levels - 1; level >= 0; --level) {
    for (int i = 0; i <= c.num_res_blocks[level]; ++i) {
      const int ich = chans.back(); chans.pop_back();
      std::vector<Layer> layers{{1, ch + ich, mc * c.channel_mult[level]}};
      ch = mc * c.channel_mult[level];
      if (e.has_attn(ds) && i == 0) layers.push_back({2, ch, ds});
      if (level && i == c.num_res_blocks[level]) { layers.push_back({4, ch, ch}); ds *= 2; }
      t.output_blocks.push_back(layers);
    }
  }
  return t;
}

void add_param(rs_engine& e, const std::string& name, std::vector<int> shape, int role) {
  Param p; p.name = name; p.shape = std::move(shape); p.role = role;
  e.index[name] = (int)e.params.size();
  e.params.push_back(std::move(p));
}
void add_conv(rs_engine& e, const std::string& n, int cin, int cout, int k) {
  add_param(e, n + ".weight", {cout, cin, k, k}, k == 3 ? R_CONV3 : R_CONV1);
  add_param(e, n + ".bias", {cout}, R_BIAS);
}
void add_linear(rs_engine& e, const std::string& n, int cin, int cout) {
  add_param(e, n + ".weight", {cout, cin}, R_LINEAR);
  add_param(e, n + ".bias", {cout}, R_BIAS);
}
void add_gn(rs_engine& e, const std::string& n, int c) {
  add_param(e, n + ".weight", {c}, R_GN_W);
  add_param(e, n + ".bias", {c}, R_GN_B);
}

void add_layers(rs_engine& e, const std::string& prefix, const std::vector<Layer>& layers) {
  const rs_unet_config& c = e.cfg;
  for (size_t j = 0; j < layers.size(); ++j) {
    const Layer& L = layers[j];
    const std::string p = prefix + "." + std::to_string(j);
    if (L.kind == 0) {
      add_conv(e, p, L.a, L.b, 3);
    } else if (L.kind == 1) {
      add_gn(e, p + ".in_layers.0", L.a);
      add_conv(e, p + ".in_layers.2", L.a, L.b, 3);
      add_linear(e, p + ".emb_layers.1", e.time_dim(), 2 * L.b);
      add_gn(e, p + ".out_layers.0", L.b);
      add_conv(e, p + ".out_layers.3", L.b, L.b, 3);
      if (L.a != L.b) add_conv(e, p + ".skip_connection", L.a, L.b, 1);
    } else if (L.kind == 2) {
      const int E = c.swin_embed_dim, res = L.b;
      const int win = res <= c.window_size ? res : c.window_size;
      const int shift = res <= c.window_size ? 0 : c.window_size / 2;
      const int hidden = (int)(E * c.mlp_ratio);
      add_conv(e, p + ".patch_embed.proj", L.a, E, 1);
      add_conv(e, p + ".patch_unembed.proj", E, L.a, 1);
      for (int i = 0; i < c.swin_depth; ++i) {
        const std::string b = p + ".blocks." + std::to_string(i);
        if (i % 2 == 1 && shift > 0) {
          const int nw = (res / win) * (res / win);
          add_param(e, b + ".attn_mask", {nw, win * win, win * win}, R_BUF_MASK);
        }
        add_gn(e, b + ".norm1", E);
        add_param(e, b + ".attn.relative_position_bias_table", {(2 * win - 1) * (2 * win - 1), c.swin_heads}, R_RELPOS);
        add_param(e, b + ".attn.relative_position_index", {win * win, win * win}, R_BUF_RELIDX);
        add_linear(e, b + ".attn.qkv", E, 3 * E);
        add_linear(e, b + ".attn.proj", E, E);
        add_gn(e, b + ".norm2", E);
        add_conv(e, b + ".mlp.fc1", E, hidden, 1);
        add_conv(e, b + ".mlp.fc2", hidden, E, 1);
      }
    } else if (L.kind == 3) {
      add_conv(e, p + ".op", L.a, L.a, 3);
    } else if (L.kind == 4) {
      add_conv(e, p + ".conv", L.a, L.a, 3);
    }
  }
}

int build_inventory(rs_engine& e) {
  const rs_unet_config& c = e.cfg;
  add_linear(e, "time_embed.0", c.model_channels, e.time_dim());
  add_linear(e, "time_embed.2", e.time_dim(), e.time_dim());
  int fc = e.lq_in_ch(), bc = 16;
  for (int st = 0; st < e.fe_stages(); ++st) {
    add_conv(e, "feature_extractor." + std::to_string(3 * st), fc, bc, 3);
    add_conv(e, "feature_extractor." + std::to_string(3 * st + 2) + ".op", bc, 2 * bc, 3);
    bc *= 2; fc = bc;
  }
  Topology t = build_topology(e);
  for (size_t i = 0; i < t.input_blocks.size(); ++i) add_layers(e, "input_blocks." + std::to_string(i), t.input_blocks[i]);
  add_layers(e, "middle_block", t.middle);
  for (size_t i = 0; i < t.output_blocks.size(); ++i) add_layers(e, "output_blocks." + std::to_string(i), t.output_blocks[i]);
  add_gn(e, "out.0", c.channel_mult[0] * c.model_channels);
  add_conv(e, "out.2", c.channel_mult[0] * c.model_channels, c.out_channels, 3);

  // arena layout.  emb_layers weights / biases first, contiguous, in ResBlock order, so that all of
  // them form ONE [film_rows, time_dim] matrix for a single small-linear launch.
  size_t off = 0;
  const int K = e.time_dim();
  e.film_w_off = off;
  int rows = 0;
  for (Param& p : e.params) {
    if (p.role == R_LINEAR && p.name.find(".emb_layers.1.weight") != std::string::npos) {
      p.ipad = K; p.off = off; p.bytes = (size_t)p.shape[0] * K * 2;
      e.film_row_of[p.name.substr(0, p.name.size() - std::string(".emb_layers.1.weight").size())] = rows;
      rows += p.shape[0];
      off += p.bytes;
    }
  }
  e.film_rows = rows;
  off = align_up(off, 256);
  e.film_b_off = off;
  for (Param& p : e.params) {
    if (p.role == R_BIAS && p.name.find(".emb_layers.1.bias") != std::string::npos) {
      p.off = off; p.bytes = (size_t)p.shape[0] * 4; off += p.bytes;
    }
  }
  off = align_up(off, 256);
  for (Param& p : e.params) {
    if (p.bytes) continue;
    switch (p.role) {
      case R_CONV3: case R_CONV1:
        p.ipad = (p.shape[1] + 7) / 8 * 8;
        p.bytes = (size_t)p.shape[0] * p.shape[2] * p.shape[3] * p.ipad * 2; break;
      case R_LINEAR:
        p.ipad = (p.shape[1] + 7) / 8 * 8;
        p.bytes = (size_t)p.shape[0] * p.ipad * 2; break;
      case R_BIAS: case R_GN_W: case R_GN_B:
        p.bytes = (size_t)p.shape[0] * 4; break;
      case R_RELPOS:
        p.bytes = (size_t)c.swin_heads * 64 * 64 * 4; break;
      default: p.bytes = 0; break;     // buffers are derived, not stored
    }
    if (p.bytes) { p.off = off; off = align_up(off + p.bytes, 256); }
  }
  e.arena_bytes = align_up(off, 256);
  return 0;
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// plan
// ------------------------------------------------------------------------------------------------
namespace {

enum OpKind { OP_CONV, OP_GN, OP_ATTN, OP_UPSAMPLE, OP_MLP, OP_SOFTMAX, OP_FORK, OP_JOIN, OP_SWIN_ATTN, OP_VQ_ATTN };

struct Tensor {
  size_t bytes = 0;
  int first = 1 << 30, last = -1;
  size_t off = 0;
  bool persistent = false;
};

struct Op {
  OpKind kind;
  ConvDesc conv;
  GnDesc gn;
  // attention
  View a_in, a_out; const float* a_bias = nullptr; int a_shift = 0;
  // upsample
  View u_in, u_out;
  // row softmax (VQ-GAN attention): in place on s_view [rows = N*H*W][cols = C]
  View s_view; float s_scale = 1.f;
  // conv whose "weight" matrix is an activation tensor of the plan (per-image attention GEMMs), or whose INPUT is a
  // weight matrix of the arena viewed as pixels (the transposed value projection): see vq.inc
  View w_view; bool w_is_view = false;
  std::string in_param;
  // fused MLP
  MlpDesc mlp;
  // fused attention half of a Swin block (norm1 + qkv + window attention + proj + residual)
  SwinAttnDesc swin;
  // fused single-head attention of the VQ-GAN bottleneck: Q, K [N][T][C], V^T [N][C][T] -> out [N][T][C] (vq.inc)
  View vqa_q, vqa_k, vqa_vt, vqa_out;
  VqAttnDesc vqa;
  std::string blk_name;
  std::string w2_name, b2_name;
  std::string w_name, b_name, g_name;   // parameter names resolved at bind
  size_t stats_off = 0;                 // GroupNorm: offset of its (mean, M2) pair buffer inside the stats region
  int gn_index = -1;                    // GroupNorm: index of its [N][32][2] group statistics / [N] arrival counters
  bool to_f32 = false;                  // conv: writes the fp32 NCHW model output
  int split_tens = -1;                  // conv: workspace tensor holding split-K partial sums (or -1)
  int stream = 0;                       // 0: the caller's stream; k > 0: side stream k of the plan (concurrent batch slices)
  struct StatDst { int list; int op; int coff; int img_off; };
  std::vector<StatDst> stat_dst;        // conv: GroupNorm ops whose statistics this conv's epilogue produces
};

}  // namespace

struct rs_plan {
  rs_engine* e = nullptr;
  int B = 0, H = 0, W = 0, lqH = 0, lqW = 0;
  std::vector<Tensor> tensors;
  std::vector<Op> fe_ops, ops;
  std::map<std::string, View> block_out;
  // fixed regions (byte offsets in the workspace)
  size_t off_emb_sin = 0, off_emb_mid = 0, off_emb_vec = 0, off_film = 0, off_tsteps = 0, off_tables = 0;
  size_t off_stats = 0, stats_bytes = 0, off_state = 0, off_temps = 0, temps_bytes = 0;
  size_t off_gstat = 0, off_counters = 0;   // per GroupNorm: [N][32][2] floats (mean, rstd); [N] arrival counters
  int n_gn = 0;
  size_t workspace_bytes = 0;
  int max_rows = 0;          // rows of the FiLM table (max(B, 64) so a sampler with T <= 64 fits)
  uint8_t* ws = nullptr;
  View xin, lq_feat, fe_in;  // packed denoiser input, LQ feature (if a feature extractor exists), its input
  int cin_pad = 0, fe_cpad = 0;
  float* out_f32 = nullptr;  // model output (fp32 NCHW), inside the state region
  bool bound = false;
  int launches = 0;
  // Low-resolution levels (a handful of output tiles per layer at batch 16: every kernel is latency-bound and leaves most
  // SMs idle) run as `branches` independent batch slices on concurrent streams; each slice's kernels depend only on its
  // own predecessors, so two (or four) of these small kernels share the machine.  Streams / events belong to the plan;
  // fork / join are event edges, so the structure is captured into the sampler's CUDA graph as parallel branches.
  int branches = 1;
  std::vector<cudaStream_t> side;          // branches - 1 side streams
  std::vector<cudaEvent_t> ev;             // [0] fork, [k] join of side stream k
  std::vector<std::pair<int, int>> sections;   // [first, last] global op index of every concurrent section
  ~rs_plan() {
    for (cudaStream_t s : side) cudaStreamDestroy(s);
    for (cudaEvent_t e : ev) cudaEventDestroy(e);
  }
  int vq_which = -1;         // -1: denoiser plan; 0 / 1: VQ-GAN encode / decode plan (vq.inc)
  int imgH = 0, imgW = 0;    // VQ plans: image size (H, W above are the latent size)
  // The schedule tables and the FiLM table live in this plan's workspace and are shared by rs_plan_forward (FiLM rows
  // 0..B-1 for the caller's timesteps) and by every sampler of the plan (rows 0..T-1 for its schedule): whoever wrote them
  // last owns them.  A sampler re-derives them when it is not the owner or when the weights changed since (weights_epoch).
  const void* table_owner = nullptr;
  unsigned long long table_epoch = ~0ull;

  int new_tensor(size_t bytes, bool persistent = false) {
    Tensor t; t.bytes = align_up(bytes, 256); t.persistent = persistent;
    tensors.push_back(t);
    return (int)tensors.size() - 1;
  }
  View make_view(int N, int Hh, int Ww, int C, bool persistent = false) {
    View v; v.N = N; v.H = Hh; v.W = Ww; v.C = C; v.ld = C; v.off = 0;
    v.tens = new_tensor((size_t)N * Hh * Ww * C * 2, persistent);
    return v;
  }
  static View slice(const View& base, int c0, int C) {
    View v = base; v.off = base.off + c0; v.c0 = base.c0 + c0; v.C = C; return v;
  }
  static View batch(const View& base, int n0, int n) {       // images [n0, n0 + n) of the view
    View v = base; v.off = base.off + (long long)n0 * base.sN(); v.n0 = base.n0 + n0; v.N = n; return v;
  }
  void touch(const View& v, int opi) {
    if (v.tens < 0) return;
    Tensor& t = tensors[v.tens];
    t.first = std::min(t.first, opi); t.last = std::max(t.last, opi);
  }
};

namespace {

struct Builder {
  rs_plan& P;
  rs_engine& E;
  std::vector<Op>* cur;
  size_t stats_off = 0;
  int n_gn = 0;
  struct Writer { int c0; int C; int n0; int N; int list; int op; int win_slots; };
  std::map<int, std::vector<Writer>> writers;      // tensor id -> latest writers by (channel range, image range)
  int cur_stream = 0;                              // ops are tagged with the stream of the batch slice being built
  int cur_batch0 = 0;                              // ... and with its first image inside the plan's batch (per-image FiLM rows)
  static bool overlaps(const Writer& w, const View& v, int C) {
    return w.c0 < v.c0 + C && v.c0 < w.c0 + w.C && w.n0 < v.n0 + v.N && v.n0 < w.n0 + w.N;
  }
  static bool inside(const Writer& w, const View& v) {
    return w.c0 >= v.c0 && w.c0 + w.C <= v.c0 + v.C && w.n0 >= v.n0 && w.n0 + w.N <= v.n0 + v.N;
  }
  void note_writer(const View& out, int C, int win_slots = 0) {
    auto& ws = writers[out.tens];
    ws.erase(std::remove_if(ws.begin(), ws.end(), [&](const Writer& w) { return overlaps(w, out, C); }), ws.end());
    ws.push_back({out.c0, C, out.n0, out.N, list_id(), (int)cur->size() - 1, win_slots});
  }
  // producers of every (channel, image) of `in` whose epilogues can deliver GroupNorm statistics (empty: not fusable)
  std::vector<Writer> covering_writers(const View& in) {
    bool fusable = false;
    conv_tile_slots(in.H, in.W, &fusable);
    std::vector<Writer> prod;
    if (fuse_stats && fusable) {
      long long covered = 0;
      auto it = writers.find(in.tens);
      if (it != writers.end())
        for (const Writer& w : it->second)
          if (inside(w, in)) { prod.push_back(w); covered += (long long)w.C * w.N; }
      bool ok = covered == (long long)in.C * in.N;
      for (const Writer& w : prod) ok = ok && list(w.list)[w.op].stat_dst.size() < 2 && w.win_slots == prod[0].win_slots;
      if (!ok) prod.clear();
    }
    return prod;
  }
  const bool fuse_mlp = env_int("RS_MLP_FUSE", 1) && !env_is("RS_CONV_IMPL", "simt");
  // norm2 applied inside the fused MLP kernel (bit-identical to the separate pass): implemented, measured twice — with
  // every MLP CTA combining the statistics itself (round 1) and with producer-finalised statistics (profiles/r2_s2:
  // 4.73 vs 4.69 ms per step) — and not faster either way, so it stays OFF (RS_MLP_NORM_FUSE=1 enables it)
  const bool fuse_mlp_norm = env_int("RS_MLP_NORM_FUSE", 0) != 0;
  // norm1 + qkv + window attention + proj + residual as one tcgen05 kernel per Swin block (swin_attn_tc.cuh; RS_SWIN_FUSE=0:
  // four launches; RS_SWIN_IMPL=mma: the mma.sync version of the fused kernel)
  const bool fuse_swin_attn = env_int("RS_SWIN_FUSE", 1) != 0 && !env_is("RS_CONV_IMPL", "simt") && !env_is("RS_ATTN_IMPL", "simt");
  // measured in the graph (profiles/r2_s33_min_pairs.log; ms per denoise step, fused from N pairs up):
  //   batch 16: all levels 3.876, >= 9: 3.834, >= 33 (64x64 + 32x32): 3.809, >= 129 (64x64 only): 3.846, none: 3.902
  //   batch  8: all 2.920, >= 33 (64x64 + 32x32 with 64 pairs): 2.826, >= 129 (64x64 only): 2.812, none: 2.877
  //   batch  1: all 2.252, none 2.097 (64x64 = 32 pairs)
  // i.e. the fused kernel wins where its persistent CTAs cover most of the machine (>= ~100 window pairs) and loses where a
  // level is one 29-us tile on a few SMs against four small launches whose prologues overlap.
  const int fuse_swin_min_pairs = env_int("RS_SWIN_FUSE_MIN_PAIRS", 96);
  const bool fuse_stats = env_int("RS_GN_FUSE", 1) && !env_is("RS_CONV_EPI", "direct") && !env_is("RS_CONV_IMPL", "simt");
  Builder(rs_plan& p) : P(p), E(*p.e), cur(&p.ops) {}
  int list_id() const { return cur == &P.fe_ops ? 0 : 1; }
  std::vector<Op>& list(int id) { return id == 0 ? P.fe_ops : P.ops; }

  int opi() const { return (int)(P.fe_ops.size() + P.ops.size()); }

  void conv(const View& in, const std::string& name, int ksize, int stride, int cout, const View* out,
            const View* res, int act, bool out_f32 = false, int pad_lo = 1) {
    Op op; op.kind = OP_CONV;
    op.conv.in = in; op.conv.ksize = ksize; op.conv.stride = stride; op.conv.Cout = cout; op.conv.act = act;
    op.conv.pad_lo = pad_lo;
    if (out) { op.conv.out = *out; op.conv.has_out = true; } else op.conv.has_out = false;
    if (res) { op.conv.res = *res; op.conv.has_res = true; }
    op.w_name = name + ".weight"; op.b_name = name + ".bias";
    op.to_f32 = out_f32;
    if (out && !out_f32 && env_int("RS_CONV_SPLITK", 0) != 1) {       // split-K for layers with too few tiles
      const TileConfig tc = conv_preview_config(in.N, in.H, in.W, in.C, cout, ksize, stride, true);
      if (tc.splitk > 1) op.conv.allow_split = true;
      if (tc.splitk > 1 && !tc.cluster_split) {       // (cluster split-K reduces through shared memory: no scratch)
        const size_t bytes = (size_t)tc.splitk * in.N * (in.H / stride) * (in.W / stride) * cout * sizeof(float);
        op.split_tens = P.new_tensor(bytes);
        Tensor& tz = P.tensors[op.split_tens];
        tz.first = tz.last = opi();
      }
    }
    const int i = opi();
    P.touch(in, i); if (out) P.touch(*out, i); if (res) P.touch(*res, i);
    op.stream = cur_stream;
    cur->push_back(op);
    if (out && !out_f32 && out->tens >= 0) note_writer(*out, cout);   // the latest writer of this (channel, image) range
  }
  void gn(const View& in, const std::string& name, const View& out, int silu, int film_off, float eps = 1e-5f) {
    Op op; op.kind = OP_GN;
    op.gn.in = in; op.gn.out = out; op.gn.silu = silu; op.gn.film_off = film_off; op.gn.eps = eps;
    op.gn.film_n0 = cur_batch0;
    op.g_name = name;
    // can the producers' epilogues deliver the statistics?  (every channel of every image of the view written by a
    // conv / MLP of this plan)
    std::vector<Writer> prod = covering_writers(in);
    op.gn.win_slots = !prod.empty() && prod[0].win_slots;
    const int tile_slots = op.gn.win_slots ? (in.H / 8) * (in.W / 8) : conv_tile_slots(in.H, in.W);
    int chunks, rows;
    gn_chunks(in.H * in.W, in.N, &chunks, &rows);
    op.gn.fused = !prod.empty();
    op.gn.slots = op.gn.fused ? tile_slots : chunks;
    op.stats_off = stats_off;
    op.gn_index = n_gn++;
    stats_off += align_up((size_t)in.N * op.gn.slots * in.C * 2 * sizeof(float), 256);
    const int i = opi();
    P.touch(in, i); P.touch(out, i);
    op.stream = cur_stream;
    cur->push_back(op);
    for (const Writer& w : prod)
      list(w.list)[w.op].stat_dst.push_back({list_id(), (int)cur->size() - 1, w.c0 - in.c0, w.n0 - in.n0});
  }
  void attn(const View& qkv, const View& out, const std::string& blk, int shift) {
    Op op; op.kind = OP_ATTN; op.a_in = qkv; op.a_out = out; op.a_shift = shift;
    op.w_name = blk + ".attn.relative_position_bias_table";
    const int i = opi();
    P.touch(qkv, i); P.touch(out, i);
    op.stream = cur_stream;
    cur->push_back(op);
  }
  // norm_name non-empty: `in` is the un-normalised tensor and the kernel applies that GroupNorm to its X tile itself
  // (returns false, adding nothing, when the statistics cannot come from the producers' epilogues)
  bool mlp(const View& in, const std::string& name, int E, int Hd, const View& out, const View& res,
           const std::string& norm_name = std::string()) {
    Op op; op.kind = OP_MLP;
    op.mlp.in = in; op.mlp.out = out; op.mlp.res = res; op.mlp.has_res = true; op.mlp.E = E; op.mlp.Hd = Hd;
    op.w_name = name + ".fc1.weight"; op.b_name = name + ".fc1.bias";
    op.w2_name = name + ".fc2.weight"; op.b2_name = name + ".fc2.bias";
    std::vector<Writer> prod;
    if (!norm_name.empty()) {
      prod = covering_writers(in);
      if (prod.empty() || Hd < 4 * E) return false;
      op.g_name = norm_name;
      op.gn.win_slots = prod[0].win_slots;
      op.gn.in = in; op.gn.fused = true; op.gn.slots = op.gn.win_slots ? (in.H / 8) * (in.W / 8) : conv_tile_slots(in.H, in.W);
      op.stats_off = stats_off;
      op.gn_index = n_gn++;
      stats_off += align_up((size_t)in.N * op.gn.slots * in.C * 2 * sizeof(float), 256);
    }
    const int i = opi();
    P.touch(in, i); P.touch(out, i); P.touch(res, i);
    op.stream = cur_stream;
    cur->push_back(op);
    for (const Writer& w : prod)
      list(w.list)[w.op].stat_dst.push_back({list_id(), (int)cur->size() - 1, w.c0 - in.c0, w.n0 - in.n0});
    if (out.tens >= 0) note_writer(out, E);
    return true;
  }
  // x <- x + proj(window_attention(qkv(norm1(x)))) in one kernel (swin_attn_fused.cuh); false when the statistics of x
  // cannot come from its producers' epilogues
  bool swin_attn(const View& x, const std::string& blk, int heads, int shift) {
    std::vector<Writer> prod = covering_writers(x);
    if (prod.empty()) return false;
    Op op; op.kind = OP_SWIN_ATTN;
    op.swin.x = x; op.swin.y = x; op.swin.heads = heads; op.swin.shift = shift;
    op.blk_name = blk;
    op.g_name = blk + ".norm1";
    op.gn.win_slots = prod[0].win_slots;
    op.gn.in = x; op.gn.fused = true; op.gn.slots = op.gn.win_slots ? (x.H / 8) * (x.W / 8) : conv_tile_slots(x.H, x.W);
    op.stats_off = stats_off;
    op.gn_index = n_gn++;
    stats_off += align_up((size_t)x.N * op.gn.slots * x.C * 2 * sizeof(float), 256);
    const int i = opi();
    P.touch(x, i);
    op.stream = cur_stream;
    cur->push_back(op);
    for (const Writer& w : prod)
      list(w.list)[w.op].stat_dst.push_back({list_id(), (int)cur->size() - 1, w.c0 - x.c0, w.n0 - x.n0});
    if (x.tens >= 0) note_writer(x, x.C, /*win_slots=*/1);
    return true;
  }
  void upsample(const View& in, const View& out) {
    Op op; op.kind = OP_UPSAMPLE; op.u_in = in; op.u_out = out;
    const int i = opi();
    P.touch(in, i); P.touch(out, i);
    op.stream = cur_stream;
    cur->push_back(op);
  }
  void marker(OpKind k) { Op op; op.kind = k; cur->push_back(op); }

  // ResBlock (reference models/unet.py:186-206)
  void res_block(const View& x, const std::string& p, int cout, const View& out) {
    View t1 = P.make_view(x.N, x.H, x.W, x.C);
    gn(x, p + ".in_layers.0", t1, 1, -1);
    View h1 = P.make_view(x.N, x.H, x.W, cout);
    conv(t1, p + ".in_layers.2", 3, 1, cout, &h1, nullptr, ACT_NONE);
    View t2 = P.make_view(x.N, x.H, x.W, cout);
    gn(h1, p + ".out_layers.0", t2, 1, E.film_row_of.at(p));
    if (x.C != cout) {
      conv(x, p + ".skip_connection", 1, 1, cout, &out, nullptr, ACT_NONE);
      conv(t2, p + ".out_layers.3", 3, 1, cout, &out, &out, ACT_NONE);     // in-place accumulate
    } else {
      conv(t2, p + ".out_layers.3", 3, 1, cout, &out, &x, ACT_NONE);
    }
  }
  // BasicLayer (reference models/swin_transformer.py:427-442) with SwinTransformerBlock.forward (:238-281)
  int basic_layer(const View& x, const std::string& p, int ctor_res, const View& out) {
    const rs_unet_config& c = E.cfg;
    const int Ed = c.swin_embed_dim, hidden = (int)(Ed * c.mlp_ratio);
    const int win = ctor_res <= c.window_size ? ctor_res : c.window_size;
    RS_CHECK(win == 8 && x.H % 8 == 0 && x.W % 8 == 0, "the window-attention kernel covers 8x8 windows only");
    const int shift_odd = ctor_res <= c.window_size ? 0 : c.window_size / 2;
    View e = P.make_view(x.N, x.H, x.W, Ed);
    conv(x, p + ".patch_embed.proj", 1, 1, Ed, &e, nullptr, ACT_NONE);
    for (int i = 0; i < c.swin_depth; ++i) {
      const std::string b = p + ".blocks." + std::to_string(i);
      // x = x + proj(attn(qkv(norm1(x)))): one kernel (swin_attn_fused.cuh), or the four-launch sequence
      // (a level with few window pairs is one long serial tile per CTA on a handful of SMs: below fuse_swin_min_pairs the
      //  four small launches, whose prologues overlap through PDL, are faster in the graph)
      const int win_pairs = (x.N * (x.H / 8) * (x.W / 8) + 1) / 2;
      if (!(fuse_swin_attn && win_pairs >= fuse_swin_min_pairs && swin_attn_supported(Ed, c.swin_heads, x.H, x.W) &&
            swin_attn(e, b, c.swin_heads, (i % 2) ? shift_odd : 0))) {
        View n1 = P.make_view(x.N, x.H, x.W, Ed);
        gn(e, b + ".norm1", n1, 0, -1);
        View qkv = P.make_view(x.N, x.H, x.W, 3 * Ed);
        conv(n1, b + ".attn.qkv", 1, 1, 3 * Ed, &qkv, nullptr, ACT_NONE);
        View a = P.make_view(x.N, x.H, x.W, Ed);
        attn(qkv, a, b, (i % 2) ? shift_odd : 0);
        conv(a, b + ".attn.proj", 1, 1, Ed, &e, &e, ACT_NONE);              // x = shortcut + attn
      }
      const bool mlp_ok = fuse_mlp && mlp_supported(Ed, hidden, x.H, x.W, x.N);
      // x = x + fc2(gelu(fc1(norm2(x)))) in one kernel, norm2 applied to the X tile in shared memory
      if (mlp_ok && fuse_mlp_norm && mlp(e, b + ".mlp", Ed, hidden, e, e, b + ".norm2")) continue;
      View n2 = P.make_view(x.N, x.H, x.W, Ed);
      gn(e, b + ".norm2", n2, 0, -1);
      if (mlp_ok) {
        mlp(n2, b + ".mlp", Ed, hidden, e, e);                            // x = x + fc2(gelu(fc1(n2))), one kernel
      } else {
        View f = P.make_view(x.N, x.H, x.W, hidden);
        conv(n2, b + ".mlp.fc1", 1, 1, hidden, &f, nullptr, ACT_GELU);
        conv(f, b + ".mlp.fc2", 1, 1, Ed, &e, &e, ACT_NONE);              // x = x + mlp
      }
    }
    conv(e, p + ".patch_unembed.proj", 1, 1, x.C, &out, nullptr, ACT_NONE);
    return 0;
  }

  int run_block(View h, const std::string& prefix, const std::vector<Layer>& layers, const View& dest, View* result) {
    for (size_t j = 0; j < layers.size(); ++j) {
      const Layer& L = layers[j];
      const std::string p = prefix + "." + std::to_string(j);
      const bool last = (j + 1 == layers.size());
      View out;
      if (L.kind == 0) {
        out = last ? dest : P.make_view(h.N, h.H, h.W, L.b);
        conv(h, p, 3, 1, L.b, &out, nullptr, ACT_NONE);
      } else if (L.kind == 1) {
        out = last ? dest : P.make_view(h.N, h.H, h.W, L.b);
        res_block(h, p, L.b, out);
      } else if (L.kind == 2) {
        out = last ? dest : P.make_view(h.N, h.H, h.W, h.C);
        int rc = basic_layer(h, p, L.b, out); if (rc) return rc;
      } else if (L.kind == 3) {
        out = dest;
        conv(h, p + ".op", 3, 2, L.a, &out, nullptr, ACT_NONE);
      } else {
        View u = P.make_view(h.N, 2 * h.H, 2 * h.W, h.C);
        upsample(h, u);
        out = dest;
        conv(u, p + ".conv", 3, 1, L.a, &out, nullptr, ACT_NONE);
      }
      h = out;
    }
    *result = h;
    return 0;
  }
};

// Workspace layout shared by the denoiser plan and the VQ-GAN plans (vq.inc): fixed regions, then persistent tensors,
// then liveness-packed temporaries.  `state_bytes` = one fp32 latent / output image; the denoiser keeps two (x_t, model out).
int finish_layout(rs_plan& P, Builder& b, size_t state_bytes, bool unet) {
  rs_engine& E = *P.e;
  const rs_unet_config& c = E.cfg;
  const int B = P.B;
  P.max_rows = std::max(B, 64);
  size_t off = 0;
  auto region = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
  if (unet) {
    P.off_tables = region(4 * 1024 * sizeof(float));                   // coef1, coef2, std, in_scale (<= 1024 steps)
    P.off_tsteps = region((size_t)P.max_rows * sizeof(float));
    P.off_emb_sin = region((size_t)P.max_rows * c.model_channels * sizeof(float));
    P.off_emb_mid = region((size_t)P.max_rows * E.time_dim() * sizeof(float));
    P.off_emb_vec = region((size_t)P.max_rows * E.time_dim() * sizeof(float));
    P.off_film = region((size_t)P.max_rows * E.film_rows * sizeof(float));
  }
  P.stats_bytes = b.stats_off;
  P.off_stats = region(P.stats_bytes);
  P.n_gn = b.n_gn;
  P.off_gstat = region((size_t)P.n_gn * B * 32 * 2 * sizeof(float));
  P.off_counters = region((size_t)P.n_gn * B * sizeof(unsigned int));
  // sampler state: x_t (fp32), model output / pred_xstart (fp32)
  const size_t lat = state_bytes;
  P.off_state = region(2 * align_up(lat, 256));
  // persistent tensors first, then liveness-packed temporaries (RS_NO_REUSE=1 keeps every tensor
  // alive for the whole forward so that rs_plan_probe can read any block output afterwards)
  // tensors born or last used inside a concurrent section stay allocated for the whole section: its batch slices run
  // on different streams, so "op index order" no longer implies "executed before"
  for (const auto& sec : P.sections)
    for (Tensor& tz : P.tensors) {
      if (tz.last < 0) continue;
      if (tz.first >= sec.first && tz.first <= sec.second) tz.first = sec.first;
      if (tz.last >= sec.first && tz.last <= sec.second) tz.last = sec.second;
    }
  if (env_int("RS_NO_REUSE", 0)) for (Tensor& tz : P.tensors) tz.persistent = true;
  for (Tensor& tz : P.tensors) if (tz.persistent) tz.off = region(tz.bytes);
  P.off_temps = off;
  {
    struct Live { size_t off, bytes; int last; };
    std::vector<Live> live;
    std::vector<int> order;
    for (int i = 0; i < (int)P.tensors.size(); ++i) if (!P.tensors[i].persistent && P.tensors[i].last >= 0) order.push_back(i);
    std::stable_sort(order.begin(), order.end(), [&](int a, int bb) { return P.tensors[a].first < P.tensors[bb].first; });
    size_t high = 0;
    for (int id : order) {
      Tensor& tz = P.tensors[id];
      live.erase(std::remove_if(live.begin(), live.end(), [&](const Live& l) { return l.last < tz.first; }), live.end());
      std::sort(live.begin(), live.end(), [](const Live& a, const Live& bb) { return a.off < bb.off; });
      size_t pos = 0;
      for (const Live& l : live) {
        if (pos + tz.bytes <= l.off) break;
        pos = std::max(pos, l.off + l.bytes);
      }
      tz.off = P.off_temps + pos;
      live.push_back({pos, tz.bytes, tz.last});
      high = std::max(high, pos + tz.bytes);
    }
    P.temps_bytes = high;
  }
  P.workspace_bytes = align_up(P.off_temps + P.temps_bytes, 256);
  return 0;
}

int build_plan(rs_plan& P) {
  rs_engine& E = *P.e;
  const rs_unet_config& c = E.cfg;
  Topology topo = build_topology(E);
  Builder b(P);
  const int B = P.B;

  // ---- feature extractor (reference models/unet.py:689-702), hoisted out of the sampling loop ----
  const int fes = E.fe_stages();
  P.lqH = P.H << fes; P.lqW = P.W << fes;
  if (fes > 0) {
    b.cur = &P.fe_ops;
    P.fe_cpad = 8;
    P.fe_in = P.make_view(B, P.lqH, P.lqW, P.fe_cpad, true);
    View cur = P.fe_in;
    int bc = 16;
    for (int st = 0; st < fes; ++st) {
      View a = P.make_view(B, cur.H, cur.W, bc, true);
      b.conv(cur, "feature_extractor." + std::to_string(3 * st), 3, 1, bc, &a, nullptr, ACT_SILU);
      View d = P.make_view(B, cur.H / 2, cur.W / 2, 2 * bc, true);
      b.conv(a, "feature_extractor." + std::to_string(3 * st + 2) + ".op", 3, 2, 2 * bc, &d, nullptr, ACT_NONE);
      cur = d; bc *= 2;
    }
    P.lq_feat = cur;
    b.cur = &P.ops;
  }

  // ---- main body -----------------------------------------------------------------------------
  const int cin = c.in_channels + E.lq_feat_ch();
  P.cin_pad = (cin + 7) / 8 * 8;
  P.xin = P.make_view(B, P.H, P.W, P.cin_pad, true);

  // concat buffers of the decoder: output block j reads cat([h, hs[n_in-1-j]])
  const int n_in = (int)topo.input_blocks.size();
  const int n_out = (int)topo.output_blocks.size();
  RS_CHECK(n_in == n_out, "encoder/decoder block counts differ");
  // resolutions of the encoder outputs
  std::vector<int> in_h(n_in), in_w(n_in);
  {
    int hh = P.H, ww = P.W;
    for (int i = 0; i < n_in; ++i) {
      for (const Layer& L : topo.input_blocks[i]) if (L.kind == 3) { hh /= 2; ww /= 2; }
      in_h[i] = hh; in_w[i] = ww;
    }
  }
  std::vector<View> cat(n_out);
  for (int j = 0; j < n_out; ++j) {
    const int k = n_in - 1 - j;
    const int ctot = topo.output_blocks[j][0].a;       // ch + ich
    cat[j] = P.make_view(B, in_h[k], in_w[k], ctot);
  }
  // ---- concurrent batch slices for the few-tile levels (see rs_plan::branches) --------------------------------
  // (measured, profiles/r2_s3: 2 slices 4.34 ms / step, 4 slices 4.76 ms against 3.90 ms for the plain sequence — the
  // tile planner re-splits every half-batch layer until it fills the machine again, so the slices do not actually share
  // it and only the launch count doubles.  Kept selectable, OFF by default.)
  {
    int nb = env_int("RS_LOWRES_STREAMS", 1);
    if (nb < 1) nb = 1;
    while (nb > 1 && (B % nb != 0 || B / nb < 1)) --nb;
    P.branches = nb;
  }
  const long long low_tiles = env_int("RS_LOWRES_TILES", 64);       // a level is "few-tile" when batch * H * W / 128 <= this
  auto is_low = [&](int hh, int ww) { return (long long)B * hh * ww / 128 <= low_tiles; };
  bool in_sec = false;
  int sec_first = 0;
  auto leave = [&]() {
    if (!in_sec) return;
    const int last = b.opi() - 1;
    b.marker(OP_JOIN);
    P.sections.push_back({sec_first, last});
    in_sec = false;
  };
  // one block of the topology: as a whole, or as `branches` batch slices on their own streams
  auto run = [&](const View& hin, const std::string& prefix, const std::vector<Layer>& layers, const View& dest, View* hout) -> int {
    bool low = P.branches > 1 && is_low(hin.H, hin.W);
    if (P.branches > 1 && !low && layers.size() == 1 && layers[0].kind == 3) low = is_low(hin.H / 2, hin.W / 2);   // the stride-2 conv entering the section
    if (!low) {
      leave();
      return b.run_block(hin, prefix, layers, dest, hout);
    }
    if (!in_sec) { b.marker(OP_FORK); sec_first = b.opi(); in_sec = true; }
    const int per = B / P.branches;
    for (int k = 0; k < P.branches; ++k) {
      View tmp;
      b.cur_stream = k; b.cur_batch0 = k * per;
      int rc = b.run_block(rs_plan::batch(hin, k * per, per), prefix, layers, rs_plan::batch(dest, k * per, per), &tmp);
      b.cur_stream = 0; b.cur_batch0 = 0;
      if (rc) return rc;
    }
    *hout = dest;
    return 0;
  };
  // encoder
  View h = P.xin;
  for (int i = 0; i < n_in; ++i) {
    const int j = n_in - 1 - i;
    const int ich = topo.in_block_ch[i];
    View dest = rs_plan::slice(cat[j], cat[j].C - ich, ich);
    // the input view of the first conv must expose the padded channel count (weights are zero-padded)
    View hin = h;
    int rc = run(hin, "input_blocks." + std::to_string(i), topo.input_blocks[i], dest, &h);
    if (rc) return rc;
    P.block_out["input_blocks." + std::to_string(i)] = h;
  }
  // middle: writes into the h-slice of cat[0]
  {
    View dest = rs_plan::slice(cat[0], 0, cat[0].C - topo.in_block_ch[n_in - 1]);
    int rc = run(h, "middle_block", topo.middle, dest, &h); if (rc) return rc;
    P.block_out["middle_block"] = h;
  }
  // decoder
  View final_h;
  for (int j = 0; j < n_out; ++j) {
    View dest;
    if (j + 1 < n_out) {
      const int ich_next = topo.in_block_ch[n_in - 2 - j];
      dest = rs_plan::slice(cat[j + 1], 0, cat[j + 1].C - ich_next);
    } else {
      const Layer& L0 = topo.output_blocks[j][0];
      dest = P.make_view(B, cat[j].H, cat[j].W, L0.b);
    }
    int rc = run(cat[j], "output_blocks." + std::to_string(j), topo.output_blocks[j], dest, &h);
    if (rc) return rc;
    P.block_out["output_blocks." + std::to_string(j)] = h;
    final_h = h;
  }
  leave();
  // head (reference models/unet.py:859-863,894)
  View t = P.make_view(B, final_h.H, final_h.W, final_h.C);
  b.gn(final_h, "out.0", t, 1, -1);
  b.conv(t, "out.2", 3, 1, c.out_channels, nullptr, nullptr, ACT_NONE, /*out_f32=*/true);

  return finish_layout(P, b, (size_t)B * std::max(c.in_channels, c.out_channels) * P.H * P.W * sizeof(float), true);
}

void resolve(rs_plan& P, View& v) {
  if (v.tens >= 0) v.ptr = reinterpret_cast<__half*>(P.ws + P.tensors[v.tens].off) + v.off;
}

// statistics destination of a producer: the consuming GroupNorm's pair buffer (+ group statistics / arrival counters)
// (img_off: a producer that covers only images [img_off, ...) of the consumer — a batch slice on a side stream)
// Who reduces the (mean, M2) pairs to the image's 32 (mean, rstd)?
//   * few tile slots (the denoiser's maps, <= 32 slots): every consumer CTA combines them itself — a finalisation step on
//     the producer's tail costs more than it saves (profiles/r2_s1, r2_s2);
//   * many slots (the VQ-GAN's 128x128 / 256x256 maps, RS_GN_FINALIZE_SLOTS moves the threshold): gn_finalize_kernel, a
//     small launch in front of the consumer (default), or — RS_GN_PRODUCER_FINALIZE=1 — the last producer CTA of each
//     image (arrival counters; measured +100 us per layer on one-tile CTAs and +800 us on the persistent kernel, whose
//     CTAs all finish together so that ONE of them ends up reducing all 16 images: profiles/r2_s9_*).
bool gn_finalizes(const Op& g) {
  static const int thr = env_int("RS_GN_FINALIZE_SLOTS", 64);
  return g.gn.slots > thr && !g.gn.win_slots;      // (the fused Swin attention kernel delivers pairs only)
}
bool gn_producer_finalizes(const Op& g) {
  static const int on = env_int("RS_GN_PRODUCER_FINALIZE", 0);
  // the tcgen05 Swin attention kernel finalises its own output statistics: its CTAs own runs of consecutive windows, so
  // every image ends on a different CTA and each CTA arrives once per image (swin_attn_tc.cuh).  Implemented, tested, and
  // measured slower in the graph (3.98 vs 3.85 ms per step, profiles/r2_s28: the arrival sits on every CTA's tail), so it is
  // OFF by default (RS_SWIN_FINALIZE=1 enables it); the consumers combine the window pairs
  static const int swin_fin = env_int("RS_SWIN_FINALIZE", 0);
  if (g.gn.win_slots) return swin_fin != 0 && swin_attn_uses_tc();
  // (a GroupNorm without a fusable producer runs gn_stats_kernel, whose few CTAs per image arrive themselves)
  return gn_finalizes(g) && (on != 0 || !g.gn.fused);
}
GnSink make_sink(rs_plan& P, const Op& g, int coff, int img_off = 0, bool consumer = false) {
  GnSink s{};
  s.part = reinterpret_cast<float*>(P.ws + P.off_stats + g.stats_off) + (size_t)img_off * g.gn.slots * g.gn.in.C * 2;
  if (gn_producer_finalizes(g) || (consumer && gn_finalizes(g))) {
    s.gstat = reinterpret_cast<float*>(P.ws + P.off_gstat) + (size_t)g.gn_index * P.B * 64 + (size_t)img_off * 64;
    s.counter = reinterpret_cast<unsigned int*>(P.ws + P.off_counters) + (size_t)g.gn_index * P.B + img_off;
  }
  s.cstride = g.gn.in.C; s.coff = coff; s.expected = (unsigned)(g.gn.slots * g.gn.in.C); s.eps = g.gn.eps;
  return s;
}

int bind_ops(rs_plan& P, std::vector<Op>& ops) {
  rs_engine& E = *P.e;
  for (Op& op : ops) {
    if (op.kind == OP_CONV) {
      for (int i = 0; i < 2; ++i) {
        op.conv.sink[i] = GnSink{};
        if (i < (int)op.stat_dst.size()) {
          const Op::StatDst& sd = op.stat_dst[i];
          op.conv.sink[i] = make_sink(P, (sd.list == 0 ? P.fe_ops : P.ops)[sd.op], sd.coff, sd.img_off);
        }
      }
      ConvDesc& d = op.conv;
      resolve(P, d.in); if (d.has_out) resolve(P, d.out); if (d.has_res) resolve(P, d.res);
      if (!op.in_param.empty()) {          // the "pixels" are the rows of a weight matrix of the arena
        const Param* wp = E.find(op.in_param);
        RS_CHECK(wp != nullptr && wp->ipad == d.in.ld, "missing / mismatching parameter " + op.in_param);
        d.in.ptr = E.at<__half>(op.in_param);
      }
      if (op.w_is_view) {                  // the "weights" are an activation tensor [Cout rows][K], K-major
        resolve(P, op.w_view);
        d.wt = op.w_view.ptr; d.ipad = op.w_view.ld;
        d.bias = op.b_name.empty() ? nullptr : E.at<float>(op.b_name);
      } else {
        const Param* w = E.find(op.w_name);
        RS_CHECK(w != nullptr, "missing parameter " + op.w_name);
        d.wt = E.at<__half>(op.w_name); d.ipad = w->ipad; d.bias = E.at<float>(op.b_name);
      }
      d.out_f32 = op.to_f32 ? P.out_f32 : nullptr;
      d.partial = op.split_tens >= 0 ? reinterpret_cast<float*>(P.ws + P.tensors[op.split_tens].off) : nullptr;
      // the first conv reads the channel-padded packed input: expose the padded width to the kernel
      if (d.in.C < d.ipad && d.in.ld >= d.ipad && d.in.tens == P.xin.tens) d.in.C = d.ipad;
      if (d.in.C < d.ipad && P.fe_in.tens >= 0 && d.in.tens == P.fe_in.tens) d.in.C = d.ipad;
      int rc = conv_finalize(d); if (rc) return rc;
      P.launches += (d.prm.splitk > 1 && !d.prm.splitk_cluster) ? 2 : 1;
    } else if (op.kind == OP_GN) {
      resolve(P, op.gn.in); resolve(P, op.gn.out);
      op.gn.gamma = E.at<float>(op.g_name + ".weight"); op.gn.beta = E.at<float>(op.g_name + ".bias");
      RS_CHECK(op.gn.gamma && op.gn.beta, "missing GroupNorm parameters " + op.g_name);
      {
        const GnSink sk = make_sink(P, op, 0, 0, true);
        op.gn.part = sk.part; op.gn.gstat = sk.gstat; op.gn.counter = sk.counter;
        op.gn.finalize_kernel = op.gn.fused && gn_finalizes(op) && !gn_producer_finalizes(op);
      }
      P.launches += (op.gn.fused ? 1 : 2) + (op.gn.finalize_kernel ? 1 : 0);
    } else if (op.kind == OP_MLP) {
      MlpDesc& m = op.mlp;
      resolve(P, m.in); resolve(P, m.out); resolve(P, m.res);
      m.w1 = E.at<__half>(op.w_name); m.b1 = E.at<float>(op.b_name);
      m.w2 = E.at<__half>(op.w2_name); m.b2 = E.at<float>(op.b2_name);
      RS_CHECK(m.w1 && m.w2 && m.b1 && m.b2, "missing MLP parameters " + op.w_name);
      const Param* w1p = E.find(op.w_name); const Param* w2p = E.find(op.w2_name);
      RS_CHECK(w1p->ipad == m.E && w2p->ipad == m.Hd, "MLP weight padding");
      if (!op.g_name.empty()) {
        const GnSink sk = make_sink(P, op, 0);
        m.gn_in_gstat = sk.gstat; m.gn_in_part = sk.part; m.gn_in_slots = op.gn.slots;
        m.gn_in_gamma = E.at<float>(op.g_name + ".weight"); m.gn_in_beta = E.at<float>(op.g_name + ".bias");
        RS_CHECK(m.gn_in_gamma && m.gn_in_beta, "missing GroupNorm parameters " + op.g_name);
      }
      for (int i = 0; i < 2; ++i) {
        m.sink[i] = GnSink{};
        if (i < (int)op.stat_dst.size()) {
          const Op::StatDst& sd = op.stat_dst[i];
          m.sink[i] = make_sink(P, (sd.list == 0 ? P.fe_ops : P.ops)[sd.op], sd.coff, sd.img_off);
        }
      }
      int rc = mlp_finalize(m); if (rc) return rc;
      ++P.launches;
    } else if (op.kind == OP_ATTN) {
      resolve(P, op.a_in); resolve(P, op.a_out);
      op.a_bias = E.at<float>(op.w_name);
      RS_CHECK(op.a_bias != nullptr, "missing " + op.w_name);
      ++P.launches;
    } else if (op.kind == OP_SWIN_ATTN) {
      SwinAttnDesc& w = op.swin;
      resolve(P, w.x); resolve(P, w.y);
      const std::string& b = op.blk_name;
      const Param* wq = E.find(b + ".attn.qkv.weight"); const Param* wp = E.find(b + ".attn.proj.weight");
      RS_CHECK(wq && wp, "missing attention parameters of " + b);
      w.wqkv = E.at<__half>(b + ".attn.qkv.weight"); w.wqkv_ld = wq->ipad; w.bqkv = E.at<float>(b + ".attn.qkv.bias");
      w.wproj = E.at<__half>(b + ".attn.proj.weight"); w.wproj_ld = wp->ipad; w.bproj = E.at<float>(b + ".attn.proj.bias");
      w.relbias = E.at<float>(b + ".attn.relative_position_bias_table");
      w.gamma = E.at<float>(b + ".norm1.weight"); w.beta = E.at<float>(b + ".norm1.bias");
      RS_CHECK(w.bqkv && w.bproj && w.relbias && w.gamma && w.beta, "missing attention parameters of " + b);
      {
        const GnSink sk = make_sink(P, op, 0);
        w.gn_part = sk.part; w.gn_slots = op.gn.slots; w.gn_gstat = sk.gstat;
      }
      for (int i = 0; i < 2; ++i) {
        w.sink[i] = GnSink{};
        if (i < (int)op.stat_dst.size()) {
          const Op::StatDst& sd = op.stat_dst[i];
          w.sink[i] = make_sink(P, (sd.list == 0 ? P.fe_ops : P.ops)[sd.op], sd.coff, sd.img_off);
        }
      }
      int rc = swin_attn_finalize(w); if (rc) return rc;
      ++P.launches;
    } else if (op.kind == OP_VQ_ATTN) {
      resolve(P, op.vqa_q); resolve(P, op.vqa_k); resolve(P, op.vqa_vt); resolve(P, op.vqa_out);
      VqAttnDesc& d = op.vqa;
      d.q = op.vqa_q.ptr; d.k = op.vqa_k.ptr; d.vt = op.vqa_vt.ptr; d.out = op.vqa_out.ptr; d.ld_out = op.vqa_out.ld;
      d.N = op.vqa_q.N; d.T = op.vqa_q.H * op.vqa_q.W; d.C = op.vqa_q.C;
      d.bias = E.at<float>(op.b_name);
      RS_CHECK(d.bias != nullptr, "missing " + op.b_name);
      RS_CHECK(op.vqa_q.ld == d.C && op.vqa_k.ld == d.C && op.vqa_vt.ld == d.T, "fused VQ attention: dense operands");
      int rc = vq_attn_finalize(d); if (rc) return rc;
      ++P.launches;
    } else if (op.kind == OP_FORK || op.kind == OP_JOIN) {
      // stream structure only
    } else if (op.kind == OP_SOFTMAX) {
      resolve(P, op.s_view);
      RS_CHECK(op.s_view.C % 8 == 0 && op.s_view.C <= 8192 && op.s_view.ld % 8 == 0, "softmax row length");
      ++P.launches;
    } else {
      resolve(P, op.u_in); resolve(P, op.u_out);
      ++P.launches;
    }
  }
  return 0;
}

struct Prof {
  std::vector<cudaEvent_t> ev;     // pairs
  std::vector<int> kind;
  int used = 0;
  cudaEvent_t get() {
    if (used == (int)ev.size()) { cudaEvent_t e; cudaEventCreate(&e); ev.push_back(e); }
    return ev[used++];
  }
  ~Prof() { for (cudaEvent_t e : ev) cudaEventDestroy(e); }
};

// RS_SKIP_KINDS (timing ablation only — results are garbage): bit 0 conv3x3, 1 conv1x1 / linear, 2 GroupNorm, 3 window
// attention (also the fused Swin and VQ-GAN attention kernels), 4 upsample, 5 fused MLP.  The time a kernel family really costs inside the graph-replayed step is the
// difference between the full step and the step without it (per-launch events and ncu both over-state small kernels).
inline bool op_skipped(const Op& op) {
  static const int skip = env_int("RS_SKIP_KINDS", 0);
  if (!skip) return false;
  switch (op.kind) {
    case OP_CONV: return (skip >> (op.conv.ksize == 3 ? 0 : 1)) & 1;
    case OP_GN: return (skip >> 2) & 1;
    case OP_ATTN: return (skip >> 3) & 1;
    case OP_UPSAMPLE: return (skip >> 4) & 1;
    case OP_MLP: return (skip >> 5) & 1;
    case OP_SWIN_ATTN: return (skip >> 3) & 1;
    case OP_VQ_ATTN: return (skip >> 3) & 1;
    case OP_SOFTMAX: case OP_FORK: case OP_JOIN: return false;
  }
  return false;
}

int run_ops(rs_plan& P, const std::vector<Op>& ops, const float* film_base, long long film_sN, cudaStream_t st0,
            Prof* prof = nullptr) {
  const bool multi = prof == nullptr && !P.side.empty();       // per-op timing runs everything on the caller's stream
  for (const Op& op : ops) {
    int rc = 0;
    if (op.kind == OP_FORK || op.kind == OP_JOIN) {
      if (multi) {
        if (op.kind == OP_FORK) {
          RS_CUDA_OK(cudaEventRecord(P.ev[0], st0));
          for (cudaStream_t s : P.side) RS_CUDA_OK(cudaStreamWaitEvent(s, P.ev[0], 0));
        } else {
          for (size_t k = 0; k < P.side.size(); ++k) {
            RS_CUDA_OK(cudaEventRecord(P.ev[k + 1], P.side[k]));
            RS_CUDA_OK(cudaStreamWaitEvent(st0, P.ev[k + 1], 0));
          }
        }
      }
      if (prof) { cudaEventRecord(prof->get(), st0); prof->kind.push_back((int)OP_UPSAMPLE); cudaEventRecord(prof->get(), st0); }
      continue;
    }
    cudaStream_t st = (multi && op.stream > 0 && op.stream <= (int)P.side.size()) ? P.side[op.stream - 1] : st0;
    if (op_skipped(op)) { if (prof) { cudaEventRecord(prof->get(), st); prof->kind.push_back((int)op.kind); cudaEventRecord(prof->get(), st); } continue; }
    if (prof) { cudaEventRecord(prof->get(), st); prof->kind.push_back((int)op.kind); }
    switch (op.kind) {
      case OP_CONV: rc = conv_launch(op.conv, st); break;
      case OP_GN: {
        GnDesc g = op.gn;
        if (g.film_off >= 0) { g.film = film_base + g.film_off + (long long)g.film_n0 * film_sN; g.film_sN = film_sN; }
        rc = gn_launch(g, st);
        break;
      }
      case OP_MLP: rc = mlp_launch(op.mlp, st); break;
      case OP_SWIN_ATTN: rc = swin_attn_launch(op.swin, st); break;
      case OP_VQ_ATTN: rc = vq_attn_launch(op.vqa, st); break;
      case OP_ATTN:
        rc = attn_launch(op.a_in, op.a_out, op.a_bias, P.e->cfg.swin_heads, P.e->cfg.swin_embed_dim, op.a_shift, st);
        break;
      case OP_SOFTMAX: {
        SoftmaxParams sp{op.s_view.ptr, (long long)op.s_view.ld, op.s_view.N * op.s_view.H * op.s_view.W, op.s_view.C, op.s_scale};
        (void)launch_k(softmax_rows_kernel, dim3((unsigned)sp.rows), dim3(256), (size_t)0, st, sp);
        if (cudaGetLastError() != cudaSuccess) rc = fail(-2, "softmax launch failed");
        break;
      }
      case OP_UPSAMPLE: {
        UpsampleParams u{op.u_in.ptr, op.u_in.sN(), op.u_in.ld, op.u_out.ptr, op.u_in.N, op.u_in.H, op.u_in.W, op.u_in.C};
        const long long total = (long long)u.N * 4 * u.H * u.W * (u.C / 8);
        (void)launch_k(upsample2x_kernel, dim3((unsigned)std::min<long long>((total + 255) / 256, 148 * 16)), dim3(256), (size_t)(0), st, u);
        if (cudaGetLastError() != cudaSuccess) rc = fail(-2, "upsample launch failed");
        break;
      }
    }
    if (prof) cudaEventRecord(prof->get(), st);
    if (rc) return rc;
  }
  return 0;
}

// timestep embedding -> time_embed MLP -> all emb_layers at once, for `rows` timesteps
int run_embedding(rs_plan& P, const float* tsteps, int rows, cudaStream_t st) {
  rs_engine& E = *P.e;
  const int mc = E.cfg.model_channels, K = E.time_dim();
  float* sinb = reinterpret_cast<float*>(P.ws + P.off_emb_sin);
  float* mid = reinterpret_cast<float*>(P.ws + P.off_emb_mid);
  float* vec = reinterpret_cast<float*>(P.ws + P.off_emb_vec);
  float* film = reinterpret_cast<float*>(P.ws + P.off_film);
  const int half = mc / 2;
  (void)launch_k(timestep_embedding_kernel, dim3((rows * half + 127) / 128), dim3(128), (size_t)(0), st, tsteps, sinb, rows, mc);
  auto lin = [&](const float* x, const __half* W, const float* bias, float* out, int Kin, int O, int si, int so) {
    const long long warps = (long long)rows * O;
    (void)launch_k(linear_small_kernel, dim3((unsigned)((warps * 32 + 255) / 256)), dim3(256), (size_t)(0), st, x, W, bias, out, rows, Kin, O, si, so);
  };
  const Param* w0 = E.find("time_embed.0.weight");
  RS_CHECK(w0 && w0->ipad == mc, "time_embed.0 layout");
  lin(sinb, E.at<__half>("time_embed.0.weight"), E.at<float>("time_embed.0.bias"), mid, mc, K, 0, 1);   // Linear -> SiLU
  lin(mid, E.at<__half>("time_embed.2.weight"), E.at<float>("time_embed.2.bias"), vec, K, K, 0, 0);
  lin(vec, reinterpret_cast<__half*>(E.arena + E.film_w_off), reinterpret_cast<float*>(E.arena + E.film_b_off), film,
      K, E.film_rows, 1, 0);                                                                              // SiLU -> Linear
  RS_CUDA_OK(cudaGetLastError());
  return 0;
}

int pack_lq_and_input(rs_plan& P, const float* x, const float* lq, const float* mask, const float* scale_tab,
                      int scale_idx, cudaStream_t st) {
  rs_engine& E = *P.e;
  const rs_unet_config& c = E.cfg;
  const long long npix = (long long)P.B * P.H * P.W;
  PackInputParams pp{};
  pp.x = x; pp.Cx = c.in_channels; pp.scale_tab = scale_tab; pp.scale_idx = scale_idx;
  pp.out = P.xin.ptr; pp.Cpad = P.cin_pad; pp.N = P.B; pp.HW = P.H * P.W;
  pp.zero_ptr = reinterpret_cast<unsigned int*>(P.ws + P.off_counters); pp.zero_n = P.n_gn * P.B;
  if (E.fe_stages() > 0) {
    RS_CHECK(!c.cond_mask || mask != nullptr, "this model is mask-conditioned: mask must be given");
    PackImageParams ip{lq, 3, c.cond_mask ? mask : nullptr, c.cond_mask ? 1 : 0, P.fe_in.ptr, P.fe_cpad, P.B, P.lqH * P.lqW};
    const long long lpix = (long long)P.B * P.lqH * P.lqW;
    (void)launch_k(pack_image_kernel, dim3((unsigned)((lpix + 255) / 256)), dim3(256), (size_t)(0), st, ip);
    int rc = run_ops(P, P.fe_ops, nullptr, 0, st); if (rc) return rc;
    pp.lq_nhwc = P.lq_feat.ptr; pp.lq_ld = P.lq_feat.ld; pp.Cl = P.lq_feat.C;
  } else {
    RS_CHECK(!c.cond_mask, "cond_mask with lq_size == image_size is not covered");
    pp.lq_nchw = lq; pp.Cl = 3;
  }
  (void)launch_k(pack_input_kernel, dim3((unsigned)((npix + 255) / 256)), dim3(256), (size_t)(0), st, pp);
  RS_CUDA_OK(cudaGetLastError());
  return 0;
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------
extern "C" {

int rs_version(void) { return 100; }
const char* rs_last_error(void) { return g_last_error.c_str(); }

int rs_unet_create(const rs_unet_config* cfg, rs_engine** out) {
  RS_CHECK(cfg && out, "null argument");
  RS_CHECK(cfg->n_levels >= 1 && cfg->n_levels <= RS_MAX_LEVELS, "n_levels");
  RS_CHECK(cfg->swin_embed_dim == cfg->swin_heads * 32, "head_dim must be 32 (num_head_channels: 32 in every shipped yaml)");
  RS_CHECK(cfg->model_channels % 32 == 0 && cfg->swin_embed_dim % 32 == 0, "GroupNorm32 needs channels % 32 == 0");
  RS_CHECK(cfg->lq_size >= cfg->image_size, "lq_size < image_size is not covered");
  auto e = std::make_unique<rs_engine>();
  e->cfg = *cfg;
  int rc = build_inventory(*e); if (rc) return rc;
  *out = e.release();
  return 0;
}
void rs_unet_destroy(rs_engine* e) { delete e; }
int rs_unet_param_count(const rs_engine* e) { return e ? (int)e->params.size() : 0; }
int rs_unet_param_info(const rs_engine* e, int index, char* name, size_t name_cap, int32_t shape[4], int32_t* ndim,
                       int32_t* is_buffer) {
  RS_CHECK(e && index >= 0 && index < (int)e->params.size(), "index out of range");
  const Param& p = e->params[index];
  if (name && name_cap) { std::strncpy(name, p.name.c_str(), name_cap - 1); name[name_cap - 1] = 0; }
  for (int i = 0; i < 4; ++i) shape[i] = i < (int)p.shape.size() ? p.shape[i] : 1;
  if (ndim) *ndim = (int)p.shape.size();
  if (is_buffer) *is_buffer = (p.role == R_BUF_RELIDX || p.role == R_BUF_MASK) ? 1 : 0;
  return 0;
}
size_t rs_unet_arena_bytes(const rs_engine* e) { return e ? e->arena_bytes : 0; }
int rs_unet_set_arena(rs_engine* e, void* arena_dev) {
  RS_CHECK(e && arena_dev && (reinterpret_cast<uintptr_t>(arena_dev) & 255) == 0, "arena must be 256-byte aligned");
  e->arena = static_cast<uint8_t*>(arena_dev);
  return 0;
}
int rs_unet_load_param(rs_engine* e, const char* name, const float* src, void* stream) {
  RS_CHECK(e && name && src, "null argument");
  RS_CHECK(e->arena != nullptr, "rs_unet_set_arena first");
  const Param* p = e->find(name);
  RS_CHECK(p != nullptr, std::string("unknown parameter ") + name);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  ++e->weights_epoch;
  if (p->bytes == 0) return 0;      // derived buffers (relative_position_index, attn_mask) are not stored
  if (p->role == R_CONV3 || p->role == R_CONV1 || p->role == R_LINEAR) {
    const int O = p->shape[0], I = p->shape[1];
    const int KH = p->shape.size() == 4 ? p->shape[2] : 1, KW = p->shape.size() == 4 ? p->shape[3] : 1;
    const long long total = (long long)O * KH * KW * p->ipad;
    (void)launch_k(pack_conv_weight_kernel, dim3((unsigned)std::min<long long>((total + 255) / 256, 4096)), dim3(256), (size_t)(0), st, 
        src, reinterpret_cast<__half*>(e->arena + p->off), O, I, KH, KW, p->ipad);
  } else if (p->role == R_RELPOS) {
    RS_CHECK(p->shape[0] == 225, "relative position table must be 15x15 (window 8)");
    (void)launch_k(expand_relpos_kernel, dim3((e->cfg.swin_heads * 4096 + 255) / 256), dim3(256), (size_t)(0), st,
        src, reinterpret_cast<float*>(e->arena + p->off), e->cfg.swin_heads);
  } else {
    long long n = 1;
    for (int v : p->shape) n *= v;
    (void)launch_k(copy_f32_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), (size_t)(0), st, src, reinterpret_cast<float*>(e->arena + p->off), n);
  }
  RS_CUDA_OK(cudaGetLastError());
  return 0;
}

int rs_plan_create(rs_engine* e, int batch, int height, int width, rs_plan** out) {
  RS_CHECK(e && out && batch > 0, "bad argument");
  RS_CHECK(e->kind == 0, "this engine is a VQ-GAN first stage: use rs_vq_plan_create");
  const int down = 1 << (e->cfg.n_levels - 1);
  RS_CHECK(height % (8 * down) == 0 && width % (8 * down) == 0,
           "latent H and W must be multiples of window_size * 2^(levels-1) (64 for the shipped configs)");
  auto p = std::make_unique<rs_plan>();
  p->e = e; p->B = batch; p->H = height; p->W = width;
  int rc = build_plan(*p); if (rc) return rc;
  *out = p.release();
  return 0;
}
void rs_plan_destroy(rs_plan* p) { delete p; }
size_t rs_plan_workspace_bytes(const rs_plan* p) { return p ? p->workspace_bytes : 0; }
int rs_plan_num_launches(const rs_plan* p) { return p ? p->launches : 0; }

int rs_plan_bind(rs_plan* p, void* workspace_dev) {
  RS_CHECK(p && workspace_dev && (reinterpret_cast<uintptr_t>(workspace_dev) & 255) == 0, "workspace must be 256-byte aligned");
  RS_CHECK(p->e->arena != nullptr, "rs_unet_set_arena before binding a plan");
  p->ws = static_cast<uint8_t*>(workspace_dev);
  if (p->vq_which >= 0) {
    p->out_f32 = reinterpret_cast<float*>(p->ws + p->off_state);
  } else {
    const size_t lat = align_up((size_t)p->B * std::max(p->e->cfg.in_channels, p->e->cfg.out_channels) * p->H * p->W * 4, 256);
    p->out_f32 = reinterpret_cast<float*>(p->ws + p->off_state + lat);
  }
  resolve(*p, p->xin);
  if (p->fe_in.tens >= 0) { resolve(*p, p->fe_in); resolve(*p, p->lq_feat); }
  for (auto& kv : p->block_out) resolve(*p, kv.second);
  p->launches = 0;
  if (p->branches > 1 && p->side.empty() && !p->sections.empty()) {
    for (int k = 1; k < p->branches; ++k) {
      cudaStream_t s = nullptr;
      RS_CUDA_OK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
      p->side.push_back(s);
    }
    for (int k = 0; k < p->branches; ++k) {
      cudaEvent_t e = nullptr;
      RS_CUDA_OK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
      p->ev.push_back(e);
    }
  }
  int rc = conv_init(); if (rc) return rc;
  rc = bind_ops(*p, p->fe_ops); if (rc) return rc;
  rc = bind_ops(*p, p->ops); if (rc) return rc;
  p->launches += p->vq_which >= 0 ? 3 : 6;   // denoiser: embedding (4) + pack (1-2); VQ: counter reset, pack / quantise, output copy
  p->bound = true;
  return 0;
}

int rs_plan_forward(rs_plan* p, const float* x, const float* timesteps, const float* lq, const float* mask, float* out,
                    void* stream) {
  RS_CHECK(p && p->bound, "plan is not bound");
  RS_CHECK(p->vq_which < 0, "this is a VQ-GAN plan: use rs_vq_encode / rs_vq_decode");
  RS_CHECK(x && timesteps && lq && out, "null tensor");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  p->table_owner = nullptr;                       // FiLM rows 0..B-1 are overwritten below
  int rc = run_embedding(*p, timesteps, p->B, st); if (rc) return rc;
  rc = pack_lq_and_input(*p, x, lq, mask, nullptr, 0, st); if (rc) return rc;
  const float* film = reinterpret_cast<const float*>(p->ws + p->off_film);
  rc = run_ops(*p, p->ops, film, p->e->film_rows, st); if (rc) return rc;
  const long long n = (long long)p->B * p->e->cfg.out_channels * p->H * p->W;
  (void)launch_k(copy_f32_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), (size_t)(0), st, p->out_f32, out, n);
  RS_CUDA_OK(cudaGetLastError());
  return 0;
}

// One forward with a CUDA-event pair around every operator; returns time per kernel family
// (ms_by_kind[0..3] = conv/linear GEMM, GroupNorm (stats+apply), window attention, upsample) and the
// algorithmic FLOPs (2*MACs on real, un-padded channels) executed by the GEMM kernels (conv / linear, fused MLP, fused
// Swin attention) in that forward.
int rs_plan_profile(rs_plan* p, const float* x, const float* timesteps, const float* lq, const float* mask,
                    double* ms_by_kind, double* conv_flops, int32_t* n_conv_launches, void* stream) {
  RS_CHECK(p && p->bound && ms_by_kind && p->vq_which < 0, "bad argument (needs a bound denoiser plan)");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  p->table_owner = nullptr;
  int rc = run_embedding(*p, timesteps, p->B, st); if (rc) return rc;
  rc = pack_lq_and_input(*p, x, lq, mask, nullptr, 0, st); if (rc) return rc;
  Prof prof;
  const float* film = reinterpret_cast<const float*>(p->ws + p->off_film);
  rc = run_ops(*p, p->ops, film, p->e->film_rows, st, &prof); if (rc) return rc;
  RS_CUDA_OK(cudaStreamSynchronize(st));
  for (int k = 0; k < 4; ++k) ms_by_kind[k] = 0.0;
  for (size_t i = 0; i < prof.kind.size(); ++i) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, prof.ev[2 * i], prof.ev[2 * i + 1]);
    const int kd = prof.kind[i];
    // (the fused Swin attention kernel is a tcgen05 GEMM kernel: qkv + QK^T + PV + proj; it counts with the GEMM family)
    ms_by_kind[(kd == (int)OP_MLP || kd == (int)OP_SWIN_ATTN) ? 0 : kd] += ms;
  }
  double fl = 0.0; int nc = 0;
  for (const Op& op : p->ops) if (op.kind == OP_MLP) {
    fl += 4.0 * (double)op.mlp.in.N * op.mlp.in.H * op.mlp.in.W * op.mlp.E * (double)op.mlp.Hd;
    ++nc;
  } else if (op.kind == OP_CONV) {
    const ConvParams& c = op.conv.prm;
    const int cin_real = op.conv.in.tens == p->xin.tens ? p->e->cfg.in_channels + p->e->lq_feat_ch() : op.conv.in.C;
    fl += 2.0 * (double)c.Nimg * c.Hout * c.Wout * c.Cout * (double)c.num_taps * cin_real;
    ++nc;
  } else if (op.kind == OP_SWIN_ATTN) {
    // per token: qkv 2 E 3E + proj 2 E E + (QK^T + PV over the 64 keys of its window) 4 * 64 * E
    const double M = (double)op.swin.x.N * op.swin.x.H * op.swin.x.W, Ed = (double)op.swin.x.C;
    fl += M * (8.0 * Ed * Ed + 256.0 * Ed);
    ++nc;
  }
  if (conv_flops) *conv_flops = fl;
  if (n_conv_launches) *n_conv_launches = nc;
  return 0;
}

// per-operator times + one-line descriptions of a profiled run_ops() pass
static void collect_profile(const rs_plan& P, const Prof& prof, double* ms, char* desc, int desc_stride, int cap, int32_t* n_ops) {
  const rs_plan* p = &P;
  const int n = std::min<int>((int)p->ops.size(), cap);
  *n_ops = n;
  for (int i = 0; i < n; ++i) {
    float t = 0.f;
    cudaEventElapsedTime(&t, prof.ev[2 * i], prof.ev[2 * i + 1]);
    ms[i] = t;
    const Op& op = p->ops[i];
    char* d = desc + (size_t)i * desc_stride;
    if (op.kind == OP_CONV) {
      const ConvParams& c = op.conv.prm;
      snprintf(d, desc_stride, "conv%dx%d s%d %dx%d Cin=%d Cout=%d grid=%d BN=%d st=%d %s", op.conv.ksize, op.conv.ksize,
               op.conv.stride, c.Hout, c.Wout, op.conv.in.C, c.Cout, op.conv.grid, c.BN, c.stages, op.w_name.c_str());
    } else if (op.kind == OP_GN) {
      snprintf(d, desc_stride, "gn %dx%d C=%d fused=%d %s", op.gn.in.H, op.gn.in.W, op.gn.in.C, (int)op.gn.fused, op.g_name.c_str());
    } else if (op.kind == OP_MLP) {
      snprintf(d, desc_stride, "mlp %dx%d E=%d Hd=%d grid=%d", op.mlp.in.H, op.mlp.in.W, op.mlp.E, op.mlp.Hd, op.mlp.grid);
    } else if (op.kind == OP_ATTN) {
      snprintf(d, desc_stride, "attn %dx%d shift=%d", op.a_in.H, op.a_in.W, op.a_shift);
    } else if (op.kind == OP_SWIN_ATTN) {
      snprintf(d, desc_stride, "swin_attn %dx%d shift=%d grid=%d", op.swin.x.H, op.swin.x.W, op.swin.shift, op.swin.grid);
    } else if (op.kind == OP_VQ_ATTN) {
      snprintf(d, desc_stride, "vq_attn %dx%d T=%d C=%d grid=%ux%ux%u", op.vqa_q.H, op.vqa_q.W, op.vqa.T, op.vqa.C, op.vqa.grid.x,
               op.vqa.grid.y, op.vqa.grid.z);
    } else if (op.kind == OP_FORK || op.kind == OP_JOIN) {
      snprintf(d, desc_stride, "%s", op.kind == OP_FORK ? "fork" : "join");
    } else if (op.kind == OP_SOFTMAX) {
      snprintf(d, desc_stride, "softmax %d", op.s_view.C);
    } else {
      snprintf(d, desc_stride, "upsample %dx%d C=%d", op.u_in.H, op.u_in.W, op.u_in.C);
    }
  }
}

// Per-operator timing of one forward: fills ms[i] and a short description for each op of the main program.
int rs_plan_profile_ops(rs_plan* p, const float* x, const float* timesteps, const float* lq, const float* mask,
                        double* ms, char* desc, int desc_stride, int cap, int32_t* n_ops, void* stream) {
  RS_CHECK(p && p->bound && ms && desc && n_ops, "bad argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  p->table_owner = nullptr;
  int rc = run_embedding(*p, timesteps, p->B, st); if (rc) return rc;
  rc = pack_lq_and_input(*p, x, lq, mask, nullptr, 0, st); if (rc) return rc;
  Prof prof;
  const float* film = reinterpret_cast<const float*>(p->ws + p->off_film);
  rc = run_ops(*p, p->ops, film, p->e->film_rows, st, &prof); if (rc) return rc;
  RS_CUDA_OK(cudaStreamSynchronize(st));
  collect_profile(*p, prof, ms, desc, desc_stride, cap, n_ops);
  return 0;
}

__global__ void probe_kernel(const __half* src, long long sN, int ld, float* dst, int N, int HW, int C) {
  pdl_trigger();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)N * C * HW) return;
  const int hw = (int)(i % HW); const int c = (int)((i / HW) % C); const int n = (int)(i / ((long long)HW * C));
  dst[i] = __half2float(src[n * sN + (long long)hw * ld + c]);
}

int rs_plan_probe(rs_plan* p, const char* block, float* dst, int32_t* channels, int32_t* h, int32_t* w, void* stream) {
  RS_CHECK(p && p->bound && block, "bad argument");
  auto it = p->block_out.find(block);
  RS_CHECK(it != p->block_out.end(), std::string("unknown block ") + block);
  const View& v = it->second;
  if (channels) *channels = v.C; if (h) *h = v.H; if (w) *w = v.W;
  if (dst) {
    const long long n = (long long)v.N * v.C * v.H * v.W;
    (void)launch_k(probe_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), (size_t)(0), static_cast<cudaStream_t>(stream), v.ptr, v.sN(), v.ld, dst, v.N, v.H * v.W, v.C);
    RS_CUDA_OK(cudaGetLastError());
  }
  return 0;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// sampler
// ------------------------------------------------------------------------------------------------
struct rs_sampler {
  rs_plan* p = nullptr;
  int T = 0;
  double kappa = 0;
  std::vector<float> coef1, coef2, stdv, in_scale, tsteps;
  float prior_coef = 0;
  float* tap_pred = nullptr; float* tap_sample = nullptr;
  cudaGraphExec_t graph = nullptr;
  cudaStream_t cap_stream = nullptr;     // capture happens on a private stream (the legacy default stream cannot capture)
  const void* g_zy = nullptr; const void* g_noise = nullptr; const void* g_lq = nullptr; const void* g_mask = nullptr;
  void* g_out = nullptr;
};

namespace {

int sampler_enqueue(rs_sampler& S, const float* z_y, const float* noises, const float* lq, const float* mask,
                    float* out_latent, cudaStream_t st) {
  rs_plan& P = *S.p;
  const rs_unet_config& c = P.e->cfg;
  RS_CHECK(c.in_channels == c.out_channels, "predict_type xstart needs out_channels == in_channels");
  const long long numel = (long long)P.B * c.in_channels * P.H * P.W;
  const size_t lat = align_up((size_t)numel * 4, 256);
  float* x_t = reinterpret_cast<float*>(P.ws + P.off_state);
  float* tab = reinterpret_cast<float*>(P.ws + P.off_tables);
  const float* coef1 = tab, *coef2 = tab + 1024, *stdv = tab + 2048, *in_scale = tab + 3072;
  (void)lat;
  // x_T = z_y + kappa * sqrt_eta_T * noise_0   (prior_sample)
  (void)launch_k(prior_sample_kernel, dim3((unsigned)((numel + 255) / 256)), dim3(256), (size_t)(0), st, z_y, noises, x_t, S.prior_coef, numel);
  // LQ feature (once) + first packed input, scaled by in_scale[T-1]
  int rc = pack_lq_and_input(P, x_t, lq, mask, in_scale, S.T - 1, st); if (rc) return rc;
  const float* film_all = reinterpret_cast<const float*>(P.ws + P.off_film);
  for (int k = 0; k < S.T; ++k) {
    const int t = S.T - 1 - k;
    rc = run_ops(P, P.ops, film_all + (long long)t * P.e->film_rows, 0, st); if (rc) return rc;
    PSampleParams pp{};
    pp.x_t = x_t; pp.x0 = P.out_f32; pp.noise = noises + (long long)(k + 1) * numel;
    pp.x_next = (t == 0) ? out_latent : x_t;
    pp.coef1 = coef1; pp.coef2 = coef2; pp.stdv = stdv; pp.in_scale = in_scale; pp.t = t;
    pp.N = P.B; pp.C = c.in_channels; pp.HW = P.H * P.W;
    pp.next_in = P.xin.ptr; pp.next_cpad = P.cin_pad;
    pp.zero_ptr = reinterpret_cast<unsigned int*>(P.ws + P.off_counters); pp.zero_n = P.n_gn * P.B;
    if (S.tap_pred) RS_CUDA_OK(cudaMemcpyAsync(S.tap_pred + (long long)k * numel, P.out_f32, numel * 4, cudaMemcpyDeviceToDevice, st));
    (void)launch_k(p_sample_kernel, dim3((unsigned)((numel + 255) / 256)), dim3(256), (size_t)(0), st, pp);
    if (S.tap_sample) RS_CUDA_OK(cudaMemcpyAsync(S.tap_sample + (long long)k * numel, pp.x_next, numel * 4, cudaMemcpyDeviceToDevice, st));
  }
  RS_CUDA_OK(cudaGetLastError());
  return 0;
}

int sampler_prepare(rs_sampler& S, cudaStream_t st) {
  // tables + the FiLM table of all T steps (depends on the timestep only: reference models/unet.py:874,
  // models/respace.py:60-63) — computed once, outside any graph capture.
  rs_plan& P = *S.p;
  if (P.table_owner == &S && P.table_epoch == P.e->weights_epoch) return 0;
  float* tab = reinterpret_cast<float*>(P.ws + P.off_tables);
  RS_CUDA_OK(cudaMemcpyAsync(tab, S.coef1.data(), S.T * 4, cudaMemcpyHostToDevice, st));
  RS_CUDA_OK(cudaMemcpyAsync(tab + 1024, S.coef2.data(), S.T * 4, cudaMemcpyHostToDevice, st));
  RS_CUDA_OK(cudaMemcpyAsync(tab + 2048, S.stdv.data(), S.T * 4, cudaMemcpyHostToDevice, st));
  RS_CUDA_OK(cudaMemcpyAsync(tab + 3072, S.in_scale.data(), S.T * 4, cudaMemcpyHostToDevice, st));
  float* ts = reinterpret_cast<float*>(P.ws + P.off_tsteps);
  RS_CUDA_OK(cudaMemcpyAsync(ts, S.tsteps.data(), S.T * 4, cudaMemcpyHostToDevice, st));
  int rc = run_embedding(P, ts, S.T, st); if (rc) return rc;
  RS_CUDA_OK(cudaStreamSynchronize(st));     // host vectors must outlive the copies; one-time setup cost
  P.table_owner = &S; P.table_epoch = P.e->weights_epoch;
  return 0;
}

}  // namespace

extern "C" {

int rs_sampler_create(rs_plan* p, int steps, const double* sqrt_etas, double kappa, const int32_t* tmap, rs_sampler** out) {
  RS_CHECK(p && p->bound && sqrt_etas && out, "bad argument (plan must be bound)");
  RS_CHECK(p->vq_which < 0, "samplers are built on denoiser plans");
  RS_CHECK(steps >= 2 && steps <= p->max_rows && steps <= 1024, "steps out of range for this plan");
  auto s = std::make_unique<rs_sampler>();
  s->p = p; s->T = steps; s->kappa = kappa;
  // posterior tables in float64, cast to fp32 like _extract_into_tensor (reference models/gaussian_diffusion.py:92-105,143-161)
  std::vector<double> etas(steps), prev(steps), alpha(steps), pv(steps);
  for (int i = 0; i < steps; ++i) etas[i] = sqrt_etas[i] * sqrt_etas[i];
  for (int i = 0; i < steps; ++i) { prev[i] = i ? etas[i - 1] : 0.0; alpha[i] = etas[i] - prev[i]; pv[i] = kappa * kappa * prev[i] / etas[i] * alpha[i]; }
  s->coef1.resize(steps); s->coef2.resize(steps); s->stdv.resize(steps); s->in_scale.resize(steps); s->tsteps.resize(steps);
  for (int i = 0; i < steps; ++i) {
    const double pvc = pv[i == 0 ? 1 : i];
    s->coef1[i] = (float)(prev[i] / etas[i]);
    s->coef2[i] = (float)(alpha[i] / etas[i]);
    const float logv = (float)std::log(pvc);
    s->stdv[i] = std::exp(0.5f * logv);
    const float e32 = (float)etas[i];
    s->in_scale[i] = 1.0f / std::sqrt(e32 * (float)(kappa * kappa) + 1.0f);
    s->tsteps[i] = (float)(tmap ? tmap[i] : i);
  }
  s->prior_coef = (float)(kappa * sqrt_etas[steps - 1]);
  *out = s.release();
  return 0;
}
void rs_sampler_destroy(rs_sampler* s) {
  if (s && s->p && s->p->table_owner == s) s->p->table_owner = nullptr;
  if (s && s->graph) cudaGraphExecDestroy(s->graph);
  if (s && s->cap_stream) cudaStreamDestroy(s->cap_stream);
  delete s;
}
int rs_sampler_set_taps(rs_sampler* s, float* pred, float* sample) {
  RS_CHECK(s, "null sampler");
  s->tap_pred = pred; s->tap_sample = sample;
  if (s->graph) { cudaGraphExecDestroy(s->graph); s->graph = nullptr; }
  return 0;
}

int rs_sampler_run(rs_sampler* s, const float* z_y, const float* noises, const float* lq, const float* mask,
                   float* out_latent, int use_graph, void* stream) {
  RS_CHECK(s && z_y && noises && lq && out_latent, "null argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int rc = sampler_prepare(*s, st); if (rc) return rc;
  if (!use_graph) return sampler_enqueue(*s, z_y, noises, lq, mask, out_latent, st);
  if (s->graph && (s->g_zy != z_y || s->g_noise != noises || s->g_lq != lq || s->g_mask != mask || s->g_out != out_latent)) {
    cudaGraphExecDestroy(s->graph); s->graph = nullptr;
  }
  if (!s->graph) {
    cudaGraph_t g = nullptr;
    if (!s->cap_stream) RS_CUDA_OK(cudaStreamCreateWithFlags(&s->cap_stream, cudaStreamNonBlocking));
    RS_CUDA_OK(cudaStreamBeginCapture(s->cap_stream, cudaStreamCaptureModeThreadLocal));
    rc = sampler_enqueue(*s, z_y, noises, lq, mask, out_latent, s->cap_stream);
    cudaError_t ce = cudaStreamEndCapture(s->cap_stream, &g);
    if (rc) { if (g) cudaGraphDestroy(g); return rc; }
    RS_CUDA_OK(ce);
    RS_CUDA_OK(cudaGraphInstantiate(&s->graph, g, 0));
    cudaGraphDestroy(g);
    s->g_zy = z_y; s->g_noise = noises; s->g_lq = lq; s->g_mask = mask; s->g_out = out_latent;
  }
  RS_CUDA_OK(cudaGraphLaunch(s->graph, st));
  return 0;
}

size_t rs_sampler_staging_bytes(const rs_sampler* s) {
  if (!s) return 0;
  const rs_plan& P = *s->p;
  const rs_unet_config& c = P.e->cfg;
  const size_t lat = align_up((size_t)P.B * c.in_channels * P.H * P.W * 4, 256);
  const size_t lq = align_up((size_t)P.B * 3 * P.lqH * P.lqW * 4, 256);
  const size_t mk = align_up((size_t)P.B * 1 * P.lqH * P.lqW * 4, 256);
  return lat * (s->T + 3) + lq + mk;
}

int rs_sampler_run_host(rs_sampler* s, const float* z_y_h, const float* noises_h, const float* lq_h, const float* mask_h,
                        float* out_h, void* staging, size_t staging_bytes, int use_graph, void* stream) {
  RS_CHECK(s && z_y_h && noises_h && lq_h && out_h && staging, "null argument");
  RS_CHECK(staging_bytes >= rs_sampler_staging_bytes(s), "staging buffer too small");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const rs_plan& P = *s->p;
  const rs_unet_config& c = P.e->cfg;
  const size_t n_lat = (size_t)P.B * c.in_channels * P.H * P.W;
  const size_t lat = align_up(n_lat * 4, 256);
  const size_t n_lq = (size_t)P.B * 3 * P.lqH * P.lqW, n_mk = (size_t)P.B * P.lqH * P.lqW;
  uint8_t* base = static_cast<uint8_t*>(staging);
  float* d_zy = reinterpret_cast<float*>(base);
  float* d_out = reinterpret_cast<float*>(base + lat);
  float* d_noise = reinterpret_cast<float*>(base + 2 * lat);
  float* d_lq = reinterpret_cast<float*>(base + lat * (s->T + 3));
  float* d_mask = reinterpret_cast<float*>(base + lat * (s->T + 3) + align_up(n_lq * 4, 256));
  RS_CUDA_OK(cudaMemcpyAsync(d_zy, z_y_h, n_lat * 4, cudaMemcpyHostToDevice, st));
  RS_CUDA_OK(cudaMemcpyAsync(d_noise, noises_h, n_lat * 4 * (s->T + 1), cudaMemcpyHostToDevice, st));
  RS_CUDA_OK(cudaMemcpyAsync(d_lq, lq_h, n_lq * 4, cudaMemcpyHostToDevice, st));
  if (mask_h) RS_CUDA_OK(cudaMemcpyAsync(d_mask, mask_h, n_mk * 4, cudaMemcpyHostToDevice, st));
  int rc = rs_sampler_run(s, d_zy, d_noise, d_lq, mask_h ? d_mask : nullptr, d_out, use_graph, stream);
  if (rc) return rc;
  RS_CUDA_OK(cudaMemcpyAsync(out_h, d_out, n_lat * 4, cudaMemcpyDeviceToHost, st));
  RS_CUDA_OK(cudaStreamSynchronize(st));
  return 0;
}

__global__ void p_sample_flat_kernel(const float* x, const float* x0, const float* nz, float* out, float c1, float c2,
                                     float sd, int t0, long long n) {
  pdl_trigger();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float v = c1 * x[i] + c2 * x0[i];
  if (!t0) v += sd * nz[i];
  out[i] = v;
}
int rs_p_sample(const float* x_t, const float* x0, const float* noise, float* x_next, float c1, float c2, float sd,
                int t_is_zero, long long numel, void* stream) {
  RS_CHECK(x_t && x0 && noise && x_next && numel > 0, "bad argument");
  (void)launch_k(p_sample_flat_kernel, dim3((unsigned)((numel + 255) / 256)), dim3(256), (size_t)(0), static_cast<cudaStream_t>(stream), 
      x_t, x0, noise, x_next, c1, c2, sd, t_is_zero, numel);
  RS_CUDA_OK(cudaGetLastError());
  return 0;
}

}  // extern "C"

#include "vq.inc"
#include "ops_api.inc"
