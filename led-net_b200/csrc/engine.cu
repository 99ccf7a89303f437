// libledb200 engine: owns the folded weights and the activation workspace of one LED-Net
// (R0 trunk = DDRNet-23-slim body + two stem taps, and LEDHead), builds a launch plan per input
// shape and runs it on the caller's stream.  See include/ledb200.h for the ABI contract.
//
// Graph (eval) follows, op for op:
//   mmseg/models/backbones/ddrnet.py:121-224   (stem, 3 bilateral stages, DAPPM, final fusion)
//   mmseg/models/utils/basic_block.py:13-75, 156-221   (BasicBlock / Bottleneck)
//   mmseg/models/utils/ppm.py:12-130           (DAPPM)
//   mmseg/models/decode_heads/led_head.py:76-99 (LEDHead eval forward, pre-activation base heads)
//   mmseg/models/decode_heads/decode_head.py:241-246, 362-379 (cls_seg; patched predict_by_feat)
//   mmseg/models/segmentors/base.py:187-188    (argmax)
// Fusion rules used by the plan (no tensor is read or written more often than the graph needs):
//   * eval BatchNorm after a conv is folded into the weights/bias;
//   * ReLU, residual add (`out += residual`) and the stage-level `self.relu(x)` run in the conv
//     epilogue; where the graph needs both x and relu(x) (ddrnet.py:192-194) the epilogue stores both;
//   * BatchNorm+ReLU in FRONT of a conv (order ('norm','act','conv'): heads, DAPPM) is applied by
//     the PRODUCER of that tensor as a second epilogue output, so zero padding stays literal zero;
//   * `x += resize(...)` is one upsample+add(+ReLU) kernel; DAPPM pooling carries its BN+ReLU.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "kernels.h"

namespace ledb {

static thread_local std::string g_err;
void set_error(const std::string& m) { g_err = m; }
int fail(int code, const std::string& m) { g_err = m; return code; }

namespace {

struct HostTensor { std::vector<float> v; std::vector<int64_t> shape; };

struct ConvDef : PackedConv {  // cin .. stride from the model definition, the device side from finalize
  std::string name;          // op / debug name
  std::string wkey;          // state-dict key of conv weight
  std::string bias_key;      // conv bias key or ""
  std::string bn_after;      // BN prefix folded into the conv ("" = none)
};
struct AffineDef { std::string bn; int c = 0; float* scale = nullptr; float* shift = nullptr; };

struct Buf { std::string name; int n, h, w, c, ld; size_t off; int f16 = 0; };   // f16: holds IEEE fp16 (ladder rungs)

struct Plan;
}  // namespace
}  // namespace ledb
struct ledb200_handle;
namespace ledb {
namespace {
using OpFn = std::function<int(ledb200_handle&, Plan&, cudaStream_t)>;
enum OpKind { K_CONV_DIRECT = 0, K_CONV_TC = 1, K_UPADD = 2, K_POOL = 3, K_AFFINE = 4, K_TAIL = 5, K_LAYOUT = 6 };
// flops / bytes are ALGORITHMIC (what the layer must move or compute), see DESIGN.md section 4
struct Op {
  std::string name; OpFn fn; int kind = 0; double flops = 0, bytes = 0;
  int lane = 0;            // 0 = detail/spatial stream, 1 = context stream (bilateral branches run concurrently)
  bool wait_other = false; // this op consumes something the OTHER lane produced: join before launching
};

struct GraphEntry { std::vector<const void*> key; cudaGraphExec_t exec = nullptr; };
struct Plan {
  int kind = 0, n = 0, h = 0, w = 0;
  std::vector<GraphEntry> graphs;   // captured CUDA graphs, keyed by the caller's buffer pointers
  std::vector<Buf> bufs;
  std::vector<Op> ops;
  size_t arena = 0;
  std::map<std::string, int> by_name;
  int ho = 0, wo = 0;
};

}  // namespace
}  // namespace ledb

using namespace ledb;

struct ledb200_handle {
  ledb200_cfg cfg;
  bool finalized = false;
  std::map<std::string, HostTensor> params;
  std::vector<std::string> expected;
  std::vector<ConvDef> convs;
  std::vector<AffineDef> affs;
  std::map<std::string, int> conv_by_name, aff_by_name;
  float* pre_scale = nullptr;   // uint8 preprocessing affine [3]
  float* pre_shift = nullptr;
  std::vector<void*> dev_allocs;   // everything on the device except the convs
  char* arena = nullptr;
  size_t arena_cap = 0;
  std::map<std::string, std::unique_ptr<Plan>> plans;
  Plan* last_plan = nullptr;
  cudaStream_t cap[2] = {nullptr, nullptr};   // engine-owned streams: graph capture / eager two-lane execution
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_x[2] = {nullptr, nullptr};
  int use_graph = 1, use_lanes = 1;
  // per-call externals
  const void* ext_img = nullptr; int ext_layout = 0;
  void* ext_pred = nullptr; int ext_pred_dtype = LEDB200_U8; float* ext_logits = nullptr;
  float *ext_c5 = nullptr, *ext_x1 = nullptr, *ext_x2 = nullptr;
  const float *in_c5 = nullptr, *in_x1 = nullptr, *in_x2 = nullptr;
  float *ext_xc = nullptr, *ext_hx1 = nullptr, *ext_hx2 = nullptr;
};

namespace ledb {
namespace {

size_t esize(const ledb200_handle& e) { return e.cfg.dtype == LEDB200_BF16 ? 2 : 4; }

// ------------------------------------------------------------------ model definition
int def_conv(ledb200_handle& e, const std::string& name, const std::string& wkey, int cin, int cout, int k,
             int stride, const std::string& bn_after, const std::string& bias_key = "") {
  ConvDef d;
  d.name = name; d.wkey = wkey; d.cin = cin; d.cout = cout; d.k = k; d.stride = stride;
  d.bn_after = bn_after; d.bias_key = bias_key;
  e.expected.push_back(wkey);
  if (!bias_key.empty()) e.expected.push_back(bias_key);
  if (!bn_after.empty())
    for (const char* s : {".weight", ".bias", ".running_mean", ".running_var"}) e.expected.push_back(bn_after + s);
  e.conv_by_name[name] = (int)e.convs.size();
  e.convs.push_back(d);
  return (int)e.convs.size() - 1;
}
// mmcv ConvModule, order (conv, norm, act): keys <p>.conv.weight, <p>.bn.*
int def_cm(ledb200_handle& e, const std::string& p, int cin, int cout, int k, int stride) {
  return def_conv(e, p, p + ".conv.weight", cin, cout, k, stride, p + ".bn");
}
int def_aff(ledb200_handle& e, const std::string& bn, int c) {
  AffineDef a; a.bn = bn; a.c = c;
  for (const char* s : {".weight", ".bias", ".running_mean", ".running_var"}) e.expected.push_back(bn + s);
  e.aff_by_name[bn] = (int)e.affs.size();
  e.affs.push_back(a);
  return (int)e.affs.size() - 1;
}
void def_basic_layer(ledb200_handle& e, const std::string& p, int cin, int cout, int stride) {
  // ddrnet.py:151-180 with BasicBlock x2
  def_cm(e, p + ".0.conv1", cin, cout, 3, stride);
  def_cm(e, p + ".0.conv2", cout, cout, 3, 1);
  if (stride != 1 || cin != cout)
    def_conv(e, p + ".0.downsample", p + ".0.downsample.0.weight", cin, cout, 1, stride, p + ".0.downsample.1");
  def_cm(e, p + ".1.conv1", cout, cout, 3, 1);
  def_cm(e, p + ".1.conv2", cout, cout, 3, 1);
}
void def_bottleneck(ledb200_handle& e, const std::string& p, int cin, int ch, int stride) {
  def_cm(e, p + ".0.conv1", cin, ch, 1, 1);
  def_cm(e, p + ".0.conv2", ch, ch, 3, stride);
  def_cm(e, p + ".0.conv3", ch, ch * 2, 1, 1);
  def_conv(e, p + ".0.downsample", p + ".0.downsample.0.weight", cin, ch * 2, 1, stride, p + ".0.downsample.1");
}
// pre-activation ConvModule (norm, act, conv), bias=False: BN is an affine on the INPUT
void def_preact(ledb200_handle& e, const std::string& p, int cin, int cout, int k) {
  def_aff(e, p + ".bn", cin);
  def_conv(e, p, p + ".conv.weight", cin, cout, k, 1, "");
}

void define_model(ledb200_handle& e) {
  const int C = e.cfg.channels, P = e.cfg.ppm_channels, HC = e.cfg.head_channels, K = e.cfg.num_classes;
  const std::string b = "backbone.", h = "decode_head.";
  def_cm(e, b + "stem.0", e.cfg.in_channels, C, 3, 2);
  def_cm(e, b + "stem.1", C, C, 3, 2);
  def_basic_layer(e, b + "stem.2", C, C, 1);
  def_basic_layer(e, b + "stem.4", C, 2 * C, 2);
  def_basic_layer(e, b + "context_branch_layers.0", 2 * C, 4 * C, 2);
  def_basic_layer(e, b + "context_branch_layers.1", 4 * C, 8 * C, 2);
  def_bottleneck(e, b + "context_branch_layers.2", 8 * C, 8 * C, 2);
  def_cm(e, b + "compression_1", 4 * C, 2 * C, 1, 1);
  def_cm(e, b + "down_1", 2 * C, 4 * C, 3, 2);
  def_cm(e, b + "compression_2", 8 * C, 2 * C, 1, 1);
  def_cm(e, b + "down_2.0", 2 * C, 4 * C, 3, 2);
  def_cm(e, b + "down_2.1", 4 * C, 8 * C, 3, 2);
  def_basic_layer(e, b + "spatial_branch_layers.0", 2 * C, 2 * C, 1);
  def_basic_layer(e, b + "spatial_branch_layers.1", 2 * C, 2 * C, 1);
  def_bottleneck(e, b + "spatial_branch_layers.2", 2 * C, 2 * C, 1);
  // DAPPM (ppm.py:57-117)
  def_preact(e, b + "spp.scales.0", 16 * C, P, 1);
  for (int i = 1; i <= 4; ++i) def_preact(e, b + "spp.scales." + std::to_string(i) + ".1", 16 * C, P, 1);
  for (int i = 0; i < 4; ++i) def_preact(e, b + "spp.processes." + std::to_string(i), P, P, 3);
  def_preact(e, b + "spp.compression", 5 * P, 4 * C, 1);
  def_preact(e, b + "spp.shortcut", 16 * C, 4 * C, 1);
  // LEDHead (led_head.py:44-51, 84-99): <p>.0 = pre-act ConvModule, <p>.1 = BN folded into the conv
  auto base_head = [&](const std::string& p, int cin, int cout) {
    def_aff(e, p + ".0.bn", cin);
    def_conv(e, p, p + ".0.conv.weight", cin, cout, 3, 1, p + ".1");
  };
  base_head(h + "head", 4 * C, HC);
  base_head(h + "aux_head", 2 * C, HC);
  base_head(h + "head_x1", C, K);
  base_head(h + "head_x2", C, K);
  def_conv(e, h + "conv_seg", h + "conv_seg.weight", HC, K, 1, 1, "", h + "conv_seg.bias");
  def_conv(e, h + "aux_cls_seg", h + "aux_cls_seg.weight", HC, K, 1, 1, "", h + "aux_cls_seg.bias");
}

// ------------------------------------------------------------------ finalize (fold + upload)
int upload(ledb200_handle& e, const std::vector<float>& host, float** dev) {
  const int rc = ledb::upload(host, dev);
  if (!rc) e.dev_allocs.push_back(*dev);
  return rc;
}

const HostTensor* get(const ledb200_handle& e, const std::string& k) {
  auto it = e.params.find(k);
  return it == e.params.end() ? nullptr : &it->second;
}

int bn_affine(const ledb200_handle& e, const std::string& bn, int c, std::vector<float>& scale,
              std::vector<float>& shift) {
  const HostTensor *w = get(e, bn + ".weight"), *b = get(e, bn + ".bias"), *m = get(e, bn + ".running_mean"),
                   *v = get(e, bn + ".running_var");
  if (!w || !b || !m || !v) return fail(LEDB200_ESTATE, "missing BatchNorm parameters: " + bn);
  if ((int)w->v.size() != c || (int)b->v.size() != c || (int)m->v.size() != c || (int)v->v.size() != c)
    return fail(LEDB200_EINVAL, "BatchNorm " + bn + ": expected " + std::to_string(c) + " channels");
  scale.resize(c); shift.resize(c);
  for (int i = 0; i < c; ++i) {
    const float s = w->v[i] / std::sqrt(v->v[i] + 1e-5f);   // eps of mmcv build_norm_layer / nn.BatchNorm2d
    scale[i] = s;
    shift[i] = b->v[i] - m->v[i] * s;
  }
  return LEDB200_OK;
}

int finalize(ledb200_handle& e) {
  std::string missing;
  int nmiss = 0;
  for (auto& k : e.expected)
    if (!e.params.count(k)) { if (nmiss++ < 8) missing += (missing.empty() ? "" : ", ") + k; }
  if (nmiss) return fail(LEDB200_ESTATE, std::to_string(nmiss) + " parameters not set, e.g. " + missing);
  for (auto& d : e.convs) {
    const HostTensor* w = get(e, d.wkey);
    const size_t want = (size_t)d.cout * d.cin * d.k * d.k;
    if (w->v.size() != want)
      return fail(LEDB200_EINVAL, d.wkey + ": expected " + std::to_string(want) + " elements, got " + std::to_string(w->v.size()));
    std::vector<float> scale, shift;
    if (!d.bn_after.empty()) {
      int rc = bn_affine(e, d.bn_after, d.cout, scale, shift);
      if (rc) return rc;
    }
    const HostTensor* b = d.bias_key.empty() ? nullptr : get(e, d.bias_key);
    if (b && (int)b->v.size() != d.cout) return fail(LEDB200_EINVAL, d.bias_key + ": wrong size");
    free_conv(d);   // a finalize retried after a failure packs again
    int rc = pack_conv(w->v.data(), b ? b->v.data() : nullptr, scale.empty() ? nullptr : scale.data(),
                       shift.empty() ? nullptr : shift.data(), d);
    if (rc) return rc;
  }
  for (auto& a : e.affs) {
    std::vector<float> scale, shift;
    int rc = bn_affine(e, a.bn, a.c, scale, shift);
    if (rc) return rc;
    if ((rc = upload(e, scale, &a.scale))) return rc;
    if ((rc = upload(e, shift, &a.shift))) return rc;
  }
  std::vector<float> ps(3), pb(3);
  for (int c = 0; c < 3; ++c) { ps[c] = 1.f / e.cfg.std[c]; pb[c] = -e.cfg.mean[c] / e.cfg.std[c]; }
  int rc = upload(e, ps, &e.pre_scale);
  if (rc) return rc;
  if ((rc = upload(e, pb, &e.pre_shift))) return rc;
  e.finalized = true;
  e.params.clear();   // host copies no longer needed
  return LEDB200_OK;
}

// ------------------------------------------------------------------ plan building
struct Builder {
  ledb200_handle& e;
  Plan& p;
  int dt;
  int cur_lane = 0;
  bool pending_wait = false;
  Builder(ledb200_handle& e_, Plan& p_) : e(e_), p(p_), dt(e_.cfg.dtype) {}
  // following ops go to `l`; wait = the next op consumes a tensor produced on the other lane
  void lane(int l, bool wait = false) { cur_lane = l; pending_wait = pending_wait || wait; }
  void tag() { p.ops.back().lane = cur_lane; p.ops.back().wait_other = pending_wait; pending_wait = false; }

  int buf(const std::string& name, int n, int h, int w, int c, int ld = 0) {
    Buf b{name, n, h, w, c, ld ? ld : c, p.arena, 0};
    p.arena += ((size_t)n * h * w * b.ld * esize(e) + 255) / 256 * 256;
    p.by_name[name] = (int)p.bufs.size();
    p.bufs.push_back(b);
    return (int)p.bufs.size() - 1;
  }
  static void* ptr(ledb200_handle& e, Plan& p, int id) { return id < 0 ? nullptr : e.arena + p.bufs[id].off; }

  // One conv op on arena buffers.  aff2: affine id for the second output (-1 = plain ReLU copy)
  struct ConvOp {
    int ci, in, out, res = -1;
    bool relu = false;
    int out2 = -1, aff2 = -1, out_coff = 0, out2_coff = 0;
    bool out_f16 = false;
  };
  // Its launch arguments.  Before the arena exists (plan time) any non-null base will do: eligibility looks only at which
  // optional tensors exist, not at their addresses.
  static ConvArgs op_args(ledb200_handle& e, Plan& p, int dtype, const ConvOp& c) {
    const Buf& bi = p.bufs[c.in];
    char* base = e.arena ? e.arena : reinterpret_cast<char*>(256);
    const size_t es = dtype == LEDB200_BF16 ? 2 : 4;
    ConvArgs a = conv_args(e.convs[c.ci], bi.n, bi.h, bi.w);
    a.in = base + bi.off; a.in_dtype = dtype;
    a.in_sc = 1; a.in_sw = bi.ld; a.in_sh = (int64_t)bi.w * bi.ld; a.in_sn = (int64_t)bi.h * bi.w * bi.ld;
    if (c.out >= 0) { a.out = base + p.bufs[c.out].off + c.out_coff * es; a.out_ld = p.bufs[c.out].ld; }
    a.out_dtype = dtype;
    if (c.out2 >= 0) {
      a.out2 = base + p.bufs[c.out2].off + c.out2_coff * es; a.out2_ld = p.bufs[c.out2].ld;
      if (c.aff2 >= 0) { a.o2_scale = e.affs[c.aff2].scale + c.out2_coff; a.o2_shift = e.affs[c.aff2].shift + c.out2_coff; }
    }
    if (c.res >= 0) { a.res = base + p.bufs[c.res].off; a.res_ld = p.bufs[c.res].ld; }
    a.out_f16 = c.out_f16 ? 1 : 0;
    a.relu = c.relu ? 1 : 0;
    return a;
  }
  // would this conv run on the tensor-core kernel?
  bool conv_uses_tc(const ConvOp& c) { return conv_use_tc(op_args(e, p, dt, c), e.cfg.conv_backend); }

  int conv(const std::string& cname, int in, int out, int res = -1, bool relu = false, int out2 = -1,
           int aff2 = -1, int out_coff = 0, int out2_coff = 0, bool out_f16 = false) {
    const ConvOp c{e.conv_by_name.at(cname), in, out, res, relu, out2, aff2, out_coff, out2_coff, out_f16};
    const Buf bi = p.bufs[in];
    const ConvDef& d = e.convs[c.ci];
    const ConvArgs a = op_args(e, p, dt, c);
    const int dtype = dt;
    const bool use_tc = conv_use_tc(a, e.cfg.conv_backend);
    const double es_ = (double)esize(e), npo = (double)bi.n * a.Ho * a.Wo;
    const double flops = 2.0 * npo * d.cout * d.cin * d.k * d.k;
    // SURVEY 8(d): every tensor read once and written once.  A second, pre-activated copy of the output (x2h, DAPPM
    // inputs ...) is an implementation choice, not an algorithmic byte: the output is counted ONCE.
    const double bytes = es_ * ((double)bi.n * bi.h * bi.w * d.cin + npo * d.cout * ((out >= 0 || out2 >= 0) + (res >= 0))) +
                         es_ * (double)d.cout * d.cin * d.k * d.k;
    p.ops.push_back({cname, [=](ledb200_handle& e, Plan& p, cudaStream_t st) -> int {
      return launch_conv(op_args(e, p, dtype, c), use_tc ? 2 : 1, "engine", st);
    }, use_tc ? K_CONV_TC : K_CONV_DIRECT, flops, bytes});
    tag();
    return out;
  }
  void out_hw(const std::string& cname, int in, int& Ho, int& Wo) {
    const ConvDef& d = e.convs[e.conv_by_name.at(cname)];
    const Buf& bi = p.bufs[in];
    const int pad = d.k / 2;
    Ho = (bi.h + 2 * pad - d.k) / d.stride + 1;
    Wo = (bi.w + 2 * pad - d.k) / d.stride + 1;
  }
  int cout(const std::string& cname) { return e.convs[e.conv_by_name.at(cname)].cout; }

  // BasicBlock (basic_block.py:62-75).  relu_out: output activation (block's own `act` or the
  // stage-level nn.ReLU that follows);  dual: also store relu(out) (out stays raw).
  int basic_block(const std::string& pfx, int in, bool relu_out, bool dual, int* relu_copy = nullptr) {
    int Ho, Wo;
    out_hw(pfx + ".conv1", in, Ho, Wo);
    const int n = p.bufs[in].n, co = cout(pfx + ".conv1");
    const int t1 = buf(pfx + ".conv1", n, Ho, Wo, co);
    conv(pfx + ".conv1", in, t1, -1, true);
    int res = in;
    if (e.conv_by_name.count(pfx + ".downsample")) {
      res = buf(pfx + ".downsample", n, Ho, Wo, co);
      conv(pfx + ".downsample", in, res, -1, false);
    }
    const int o = buf(pfx, n, Ho, Wo, co);
    int o2 = -1;
    if (dual) { o2 = buf(pfx + ".relu", n, Ho, Wo, co); if (relu_copy) *relu_copy = o2; }
    conv(pfx + ".conv2", t1, o, res, relu_out, o2);
    return o;
  }
  // Bottleneck (basic_block.py:206-221), no output activation here (act_cfg_out=None in ddrnet.py)
  int bottleneck(const std::string& pfx, int in) {
    const int n = p.bufs[in].n;
    int H1, W1, H2, W2;
    out_hw(pfx + ".conv1", in, H1, W1);
    const int c1 = cout(pfx + ".conv1"), c3 = cout(pfx + ".conv3");
    const int t1 = buf(pfx + ".conv1", n, H1, W1, c1);
    conv(pfx + ".conv1", in, t1, -1, true);
    out_hw(pfx + ".conv2", t1, H2, W2);
    const int t2 = buf(pfx + ".conv2", n, H2, W2, c1);
    conv(pfx + ".conv2", t1, t2, -1, true);
    const int ds = buf(pfx + ".downsample", n, H2, W2, c3);
    conv(pfx + ".downsample", in, ds, -1, false);
    const int o = buf(pfx, n, H2, W2, c3);
    conv(pfx + ".conv3", t2, o, ds, false);
    return o;
  }
  void upadd(const std::string& name, int base, int src, int out, bool relu, int out2 = -1, int aff2 = -1) {
    const int dtype = dt;
    p.ops.push_back({name, [=](ledb200_handle& e, Plan& p, cudaStream_t st) -> int {
      UpAddArgs a;
      const Buf& bs = p.bufs[src];
      const Buf& bo = p.bufs[out >= 0 ? out : out2];
      a.base = ptr(e, p, base); a.src = ptr(e, p, src); a.out = ptr(e, p, out); a.out2 = ptr(e, p, out2);
      a.out_ld = out >= 0 ? p.bufs[out].ld : 0; a.out2_ld = out2 >= 0 ? p.bufs[out2].ld : 0;
      if (aff2 >= 0) { a.o2_scale = e.affs[aff2].scale; a.o2_shift = e.affs[aff2].shift; }
      a.dtype = dtype; a.N = bo.n; a.H = bo.h; a.W = bo.w; a.C = bs.c; a.h = bs.h; a.w = bs.w; a.relu = relu;
      return launch_upsample_add(a, st);
    }, K_UPADD, 0.0, 0.0});
    tag();
    {
      const Buf& bs = p.bufs[src];
      const Buf& bo = p.bufs[out >= 0 ? out : out2];
      const double big = (double)bo.n * bo.h * bo.w * bs.c;
      p.ops.back().bytes = esize(e) * (big * ((base >= 0) + (out >= 0 || out2 >= 0)) + (double)bs.n * bs.h * bs.w * bs.c);
      p.ops.back().flops = 8.0 * big;
    }
  }
  void pool(const std::string& name, int in, int out, int k, int s, int pd, int aff) {
    const int dtype = dt;
    p.ops.push_back({name, [=](ledb200_handle& e, Plan& p, cudaStream_t st) -> int {
      PoolArgs a;
      const Buf &bi = p.bufs[in], &bo = p.bufs[out];
      a.in = ptr(e, p, in); a.out = ptr(e, p, out); a.scale = e.affs[aff].scale; a.shift = e.affs[aff].shift;
      a.dtype = dtype; a.N = bi.n; a.H = bi.h; a.W = bi.w; a.C = bi.c; a.Ho = bo.h; a.Wo = bo.w; a.k = k; a.s = s; a.p = pd;
      return launch_avgpool_bnrelu(a, st);
    }, K_POOL, 0.0, 0.0});
    tag();
    p.ops.back().bytes = esize(e) * ((double)p.bufs[in].n * p.bufs[in].h * p.bufs[in].w * p.bufs[in].c +
                                     (double)p.bufs[out].n * p.bufs[out].h * p.bufs[out].w * p.bufs[out].c);
  }
  void affine2(const std::string& name, int in, int oa, int affa, int ob, int affb) {
    const int dtype = dt;
    p.ops.push_back({name, [=](ledb200_handle& e, Plan& p, cudaStream_t st) -> int {
      AffineArgs a;
      const Buf& bi = p.bufs[in];
      a.in = ptr(e, p, in); a.out_a = ptr(e, p, oa); a.out_b = ptr(e, p, ob);
      a.sa = e.affs[affa].scale; a.ba = e.affs[affa].shift;
      if (ob >= 0) { a.sb = e.affs[affb].scale; a.bb = e.affs[affb].shift; }
      a.dtype = dtype; a.npix = (int64_t)bi.n * bi.h * bi.w; a.C = bi.c;
      return launch_affine_relu(a, st);
    }, K_AFFINE, 0.0, 0.0});
    tag();
    p.ops.back().bytes = esize(e) * (double)p.bufs[in].n * p.bufs[in].h * p.bufs[in].w * p.bufs[in].c * (1 + (oa >= 0 || ob >= 0));
  }
};

int aff(ledb200_handle& e, const std::string& bn) { return e.aff_by_name.at(bn); }

// stem convolution 0 reads the caller's image directly (NCHW fp32, or raw uint8 with the
// SegDataPreProcessor normalisation as the conv prologue: data_preprocessor.py:112-118).
void add_stem0(Builder& B, int out_x1, int out_x1h) {
  const int dtype = B.dt;
  ledb200_handle& e0 = B.e;
  const int ci = e0.conv_by_name.at("backbone.stem.0");
  const int a2 = aff(e0, "decode_head.head_x1.0.bn");
  const int n = B.p.n, H = B.p.h, W = B.p.w;
  const int c0 = e0.convs[ci].cout;
  const bool use_tc = e0.cfg.conv_backend != 1 && dtype == LEDB200_BF16 && (c0 == 16 || c0 == 32);
  B.p.ops.push_back({"backbone.stem.0", [=](ledb200_handle& e, Plan& p, cudaStream_t st) -> int {
    ConvArgs a = conv_args(e.convs[ci], n, H, W);
    const int lay = e.ext_layout;
    const int64_t HW = (int64_t)H * W;
    a.in = e.ext_img;
    if (lay == LEDB200_IMG_NCHW_F32) {
      a.in_dtype = LEDB200_F32; a.in_sn = 3 * HW; a.in_sc = HW; a.in_sh = W; a.in_sw = 1;
    } else {
      a.in_dtype = LEDB200_U8;
      if (lay == LEDB200_IMG_NCHW_U8) { a.in_sn = 3 * HW; a.in_sc = HW; a.in_sh = W; a.in_sw = 1; }
      else { a.in_sn = 3 * HW; a.in_sc = 1; a.in_sh = 3 * (int64_t)W; a.in_sw = 3; }
      if (e.cfg.bgr_to_rgb) { a.in = (const uint8_t*)e.ext_img + 2 * a.in_sc; a.in_sc = -a.in_sc; }
      a.pre_scale = e.pre_scale; a.pre_shift = e.pre_shift; a.pre_relu = 0;
    }
    a.out = Builder::ptr(e, p, out_x1); a.out_ld = p.bufs[out_x1].ld; a.out_dtype = dtype;
    if (out_x1h >= 0) {
      a.out2 = Builder::ptr(e, p, out_x1h); a.out2_ld = p.bufs[out_x1h].ld;
      a.o2_scale = e.affs[a2].scale; a.o2_shift = e.affs[a2].shift;
    }
    a.relu = 1;
    if (use_tc && stem_tc_eligible(a)) return launch_stem_tc(a, st);
    return launch_conv_direct(a, st);
  }, use_tc ? K_CONV_TC : K_CONV_DIRECT, 0.0, 0.0});
  {
    const Buf& bo = B.p.bufs[out_x1];
    const double npo = (double)bo.n * bo.h * bo.w;
    B.p.ops.back().flops = 2.0 * npo * bo.c * 27;
    // image counted at the engine's activation width (SURVEY section 8d counts bf16 activations)
    B.p.ops.back().bytes = esize(B.e) * ((double)n * H * W * 3 + npo * bo.c);     // x1 once; the x1h copy is not credited
  }
}

enum { PLAN_INFER = 0, PLAN_BACKBONE = 1, PLAN_HEAD = 2, PLAN_HEAD_NHWC = 3 };

// Trunk: returns buffer ids through the plan's by_name map: "x1","x2","c5" (raw, optional), "c5h","x1h","x2h".
void build_trunk(Builder& B, bool raw_c5, bool head_inputs) {
  ledb200_handle& e = B.e;
  Plan& p = B.p;
  const int n = p.n, C = e.cfg.channels;
  const std::string b = "backbone.";
  const int h2 = (p.h + 2 - 3) / 2 + 1, w2 = (p.w + 2 - 3) / 2 + 1;
  const int x1 = B.buf("x1", n, h2, w2, C);
  const int x1h = head_inputs ? B.buf("x1h", n, h2, w2, C) : -1;
  add_stem0(B, x1, x1h);
  const int h4 = (h2 + 2 - 3) / 2 + 1, w4 = (w2 + 2 - 3) / 2 + 1;
  const int x2 = B.buf("x2", n, h4, w4, C);
  const int x2h = head_inputs ? B.buf("x2h", n, h4, w4, C) : -1;
  B.conv(b + "stem.1", x1, x2, -1, true, x2h, head_inputs ? aff(e, "decode_head.head_x2.0.bn") : -1);
  // layer1, layer2 (+ the nn.ReLU that follows each: ddrnet.py:140-147)
  int t = B.basic_block(b + "stem.2.0", x2, true, false);
  t = B.basic_block(b + "stem.2.1", t, true, false);
  t = B.basic_block(b + "stem.4.0", t, true, false);
  const int x = B.basic_block(b + "stem.4.1", t, true, false);
  // ---- stage 3 (ddrnet.py:190-201).  The context (lane 1) and spatial (lane 0) branches are independent
  //      between the bilateral fusion points, so they are issued on two streams: the low-resolution
  //      context convolutions have too few tiles to fill 148 SMs and overlap with the HBM-bound
  //      spatial ones.
  int xc_r = -1, xs_r = -1;
  B.lane(1, true);
  t = B.basic_block(b + "context_branch_layers.0.0", x, true, false);
  int xc = B.basic_block(b + "context_branch_layers.0.1", t, false, true, &xc_r);
  B.lane(0);
  t = B.basic_block(b + "spatial_branch_layers.0.0", x, true, false);
  int xs = B.basic_block(b + "spatial_branch_layers.0.1", t, false, true, &xs_r);
  B.lane(1);
  int comp = B.buf("comp1", n, p.bufs[xc].h, p.bufs[xc].w, 2 * C);
  B.conv(b + "compression_1", xc_r, comp);
  B.lane(0, true);
  int xs_in = B.buf("xs4in", n, p.bufs[xs].h, p.bufs[xs].w, 2 * C);
  B.upadd("fuse3.up_add", xs, comp, xs_in, true);                    // relu(x_s + up(comp_c))
  B.lane(1, true);
  int xc_in = B.buf("xc4in", n, p.bufs[xc].h, p.bufs[xc].w, 4 * C);
  B.conv(b + "down_1", xs_r, xc_in, xc, true);                       // relu(x_c + down_1(relu(x_s)))
  // ---- stage 4 (ddrnet.py:203-212)
  t = B.basic_block(b + "context_branch_layers.1.0", xc_in, true, false);
  xc = B.basic_block(b + "context_branch_layers.1.1", t, false, true, &xc_r);
  B.lane(0);
  t = B.basic_block(b + "spatial_branch_layers.1.0", xs_in, true, false);
  xs = B.basic_block(b + "spatial_branch_layers.1.1", t, false, true, &xs_r);
  B.lane(1);
  comp = B.buf("comp2", n, p.bufs[xc].h, p.bufs[xc].w, 2 * C);
  B.conv(b + "compression_2", xc_r, comp);
  B.lane(0, true);
  xs_in = B.buf("xs5in", n, p.bufs[xs].h, p.bufs[xs].w, 2 * C);
  B.upadd("fuse4.up_add", xs, comp, xs_in, true);
  B.lane(1, true);
  int Hd, Wd;
  B.out_hw(b + "down_2.0", xs_r, Hd, Wd);
  const int d2a = B.buf("down_2.0", n, Hd, Wd, 4 * C);
  B.conv(b + "down_2.0", xs_r, d2a, -1, true);
  xc_in = B.buf("xc5in", n, p.bufs[xc].h, p.bufs[xc].w, 8 * C);
  B.conv(b + "down_2.1", d2a, xc_in, xc, true);
  // ---- stage 5 (ddrnet.py:214-224): context bottleneck + DAPPM on lane 1, spatial bottleneck on lane 0
  const int xc5 = B.bottleneck(b + "context_branch_layers.2.0", xc_in);
  B.lane(0);
  const int xs5 = B.bottleneck(b + "spatial_branch_layers.2.0", xs_in);
  B.lane(1);
  // DAPPM (ppm.py:119-130)
  const int P = e.cfg.ppm_channels;
  const int hh = p.bufs[xc5].h, ww = p.bufs[xc5].w, cc = p.bufs[xc5].c;
  const std::string s = b + "spp.";
  const int ks[3] = {5, 9, 17}, ss[3] = {2, 4, 8}, ps[3] = {2, 4, 8};
  {
    // Fused DAPPM (dappm.cu): pooled branches in one launch, everything at full DAPPM resolution in one clustered
    // tcgen05 kernel - 2 launches for the module instead of 22.  bf16 engine, <= 8 tiles of 16 x 8 pixels per image.
    const bool no_fused = getenv("LEDB200_NO_FUSED_DAPPM") != nullptr;   // read per plan build: tests compare both paths
    DappmArgs probe;
    probe.N = n; probe.H = hh; probe.W = ww; probe.C = cc; probe.P = P; probe.Cout = 4 * C; probe.out_ld = 4 * C;
    if (!no_fused && B.dt == LEDB200_BF16 && e.cfg.conv_backend != 1 && dappm_eligible(probe)) {
      int sdim[4][2], sbuf[4];
      for (int i = 0; i < 4; ++i) {
        sdim[i][0] = i < 3 ? (hh + 2 * ps[i] - ks[i]) / ss[i] + 1 : 1;
        sdim[i][1] = i < 3 ? (ww + 2 * ps[i] - ks[i]) / ss[i] + 1 : 1;
        sbuf[i] = B.buf("spp.s" + std::to_string(i + 1), n, sdim[i][0], sdim[i][1], P);
      }
      const int t0 = B.buf("spp.t_even", n, hh, ww, P), t1 = B.buf("spp.t_odd", n, hh, ww, P);
      const int spp = B.buf("spp.out", n, hh, ww, 4 * C);
      auto cv = [&e, s](const std::string& name) { return e.conv_by_name.at(s + name); };
      auto af = [&e, s](const std::string& name) { return e.aff_by_name.at(s + name + ".bn"); };
      int c_scale[4], c_proc[4], a_scale[4], a_proc[4];
      for (int i = 0; i < 4; ++i) {
        c_scale[i] = cv("scales." + std::to_string(i + 1) + ".1"); a_scale[i] = af("scales." + std::to_string(i + 1) + ".1");
        c_proc[i] = cv("processes." + std::to_string(i)); a_proc[i] = af("processes." + std::to_string(i));
      }
      const int c_s0 = cv("scales.0"), c_sc = cv("shortcut"), c_comp = cv("compression");
      const int a_s0 = af("scales.0"), a_sc = af("shortcut"), a_comp = af("compression");
      const double npx = (double)n * hh * ww;
      double flops = 2.0 * npx * (2.0 * cc * P + 4.0 * 9 * P * P + 5.0 * P * 4 * C);
      double wbytes = 2.0 * (2.0 * cc * P + 4.0 * 9 * P * P + 5.0 * P * 4 * C + 4.0 * cc * P);
      for (int i = 0; i < 4; ++i) flops += 2.0 * n * sdim[i][0] * sdim[i][1] * cc * P;
      p.ops.push_back({"backbone.spp (pooled branches + fused chain)", [=](ledb200_handle& e, Plan& p, cudaStream_t st) -> int {
        DappmArgs a;
        a.x = Builder::ptr(e, p, xc5); a.N = n; a.H = hh; a.W = ww; a.C = cc; a.P = P; a.Cout = 4 * C;
        for (int i = 0; i < 4; ++i) {
          a.pool_k[i] = i < 3 ? ks[i] : 0; a.pool_s[i] = i < 3 ? ss[i] : 1; a.pool_p[i] = i < 3 ? ps[i] : 0;
          a.sh[i] = sdim[i][0]; a.sw[i] = sdim[i][1];
          a.a_scale[i] = e.affs[a_scale[i]].scale; a.b_scale[i] = e.affs[a_scale[i]].shift;
          a.w_scale[i] = e.convs[c_scale[i]].w_tc; a.bias_scale[i] = e.convs[c_scale[i]].bias;
          a.s[i] = Builder::ptr(e, p, sbuf[i]);
          a.a_proc[i] = e.affs[a_proc[i]].scale; a.b_proc[i] = e.affs[a_proc[i]].shift;
          a.w_proc[i] = e.convs[c_proc[i]].w_tc; a.bias_proc[i] = e.convs[c_proc[i]].bias;
        }
        a.a_s0 = e.affs[a_s0].scale; a.b_s0 = e.affs[a_s0].shift; a.w_s0 = e.convs[c_s0].w_tc; a.bias_s0 = e.convs[c_s0].bias;
        a.a_sc = e.affs[a_sc].scale; a.b_sc = e.affs[a_sc].shift; a.w_sc = e.convs[c_sc].w_tc; a.bias_sc = e.convs[c_sc].bias;
        a.a_comp = e.affs[a_comp].scale; a.b_comp = e.affs[a_comp].shift; a.w_comp = e.convs[c_comp].w_tc;
        a.bias_comp = e.convs[c_comp].bias;
        a.t0 = Builder::ptr(e, p, t0); a.t1 = Builder::ptr(e, p, t1);
        a.out = Builder::ptr(e, p, spp); a.out_ld = p.bufs[spp].ld;
        return launch_dappm(a, st);
      }, K_CONV_TC, flops, 2.0 * npx * (cc + 4 * C) + wbytes});
      B.tag();
      const int c5 = raw_c5 ? B.buf("c5", n, p.bufs[xs5].h, p.bufs[xs5].w, 4 * C) : -1;
      const int c5h = head_inputs ? B.buf("c5h", n, p.bufs[xs5].h, p.bufs[xs5].w, 4 * C) : -1;
      B.lane(0, true);
      B.upadd("final.up_add", xs5, spp, c5, false, c5h, head_inputs ? aff(e, "decode_head.head.0.bn") : -1);
      return;
    }
  }
  const int a0 = B.buf("spp.a0", n, hh, ww, cc), asc = B.buf("spp.asc", n, hh, ww, cc);
  B.affine2("spp.bnrelu(scales.0,shortcut)", xc5, a0, aff(e, s + "scales.0.bn"), asc, aff(e, s + "shortcut.bn"));
  const int cat = B.buf("spp.cat", n, hh, ww, 5 * P);
  const int acomp = aff(e, s + "compression.bn");
  int fprev = B.buf("spp.f0", n, hh, ww, P);
  B.conv(s + "scales.0", a0, fprev, -1, false, cat, acomp, 0, 0);
  for (int i = 1; i <= 4; ++i) {
    const std::string si = std::to_string(i);
    int ph, pw;
    if (i < 4) { ph = (hh + 2 * ps[i - 1] - ks[i - 1]) / ss[i - 1] + 1; pw = (ww + 2 * ps[i - 1] - ks[i - 1]) / ss[i - 1] + 1; }
    else { ph = 1; pw = 1; }
    const int pooled = B.buf("spp.pool" + si, n, ph, pw, cc);
    B.pool("spp.pool" + si, xc5, pooled, i < 4 ? ks[i - 1] : 0, i < 4 ? ss[i - 1] : 1, i < 4 ? ps[i - 1] : 0,
           aff(e, s + "scales." + si + ".1.bn"));
    const int sc = B.buf("spp.s" + si, n, ph, pw, P);
    B.conv(s + "scales." + si + ".1", pooled, sc);
    const int tin = B.buf("spp.t" + si, n, hh, ww, P);
    B.upadd("spp.up_add" + si, fprev, sc, -1, false, tin, aff(e, s + "processes." + std::to_string(i - 1) + ".bn"));
    const int f = (i < 4) ? B.buf("spp.f" + si, n, hh, ww, P) : -1;
    B.conv(s + "processes." + std::to_string(i - 1), tin, f, -1, false, cat, acomp, 0, i * P);
    fprev = f;
  }
  const int sp1 = B.buf("spp.comp", n, hh, ww, 4 * C);
  B.conv(s + "compression", cat, sp1);
  const int spp = B.buf("spp.out", n, hh, ww, 4 * C);
  B.conv(s + "shortcut", asc, spp, sp1, false);
  // c5 = x_s + up(spp)  (ddrnet.py:218-224); head prologue BN+ReLU fused as 2nd output
  const int c5 = raw_c5 ? B.buf("c5", n, p.bufs[xs5].h, p.bufs[xs5].w, 4 * C) : -1;
  const int c5h = head_inputs ? B.buf("c5h", n, p.bufs[xs5].h, p.bufs[xs5].w, 4 * C) : -1;
  B.lane(0, true);
  B.upadd("final.up_add", xs5, spp, c5, false, c5h, head_inputs ? aff(e, "decode_head.head.0.bn") : -1);
}

int kpad(int k) { return (k + 7) / 8 * 8; }

void build_head_fused(Builder& B) {
  ledb200_handle& e = B.e;
  Plan& p = B.p;
  const int n = p.n, K = e.cfg.num_classes, HC = e.cfg.head_channels;
  const std::string h = "decode_head.";
  const int c5h = p.by_name.at("c5h"), x1h = p.by_name.at("x1h"), x2h = p.by_name.at("x2h");
  const int hf = B.buf("head.feat", n, p.bufs[c5h].h, p.bufs[c5h].w, HC);
  B.conv(h + "head", c5h, hf, -1, true);
  const int xc = B.buf("xc", n, p.bufs[c5h].h, p.bufs[c5h].w, K, kpad(K));
  const int hx1 = B.buf("hx1", n, p.bufs[x1h].h, p.bufs[x1h].w, K, kpad(K));
  const int hx2 = B.buf("hx2", n, p.bufs[x2h].h, p.bufs[x2h].w, K, kpad(K));
  p.ho = 2 * p.bufs[hx1].h; p.wo = 2 * p.bufs[hx1].w;
  const int dtype = B.dt;
  // Ladder on the tensor cores (ladder_tc.cu): when every rung is an exact x2 (all BASELINE sizes), K <= 24 and the
  // engine runs bf16, conv_seg stores x_c in fp16, the head_x2 rung kernel forms r2 = head_x2 + up(x_c), and the head_x1
  // rung kernel forms r1 = head_x1 + up(r2), exchanges it inside the CTA and does the last x2 upsample + argmax itself:
  // neither r1 nor the full-resolution logits reach HBM.  When the caller asks for the logits, the head_x1 rung stores
  // r1 (fp16) and tail2_kernel produces logits + labels.  Otherwise (fp32 parity mode, odd sizes, K > 24) the
  // three-level tail runs.
  const bool exact2 = p.bufs[hx1].h == 2 * p.bufs[hx2].h && p.bufs[hx1].w == 2 * p.bufs[hx2].w &&
                      p.bufs[hx2].h == 2 * p.bufs[xc].h && p.bufs[hx2].w == 2 * p.bufs[xc].w;
  auto rung_args = [&e](Plan& p, const std::string& cname, int in, int up, int out) {
    const ConvDef& d = e.convs[e.conv_by_name.at(cname)];
    const Buf &bi = p.bufs[in], &bu = p.bufs[up];
    LadderArgs a;
    a.in = e.arena ? Builder::ptr(e, p, in) : (const void*)16; a.in_ld = bi.ld;
    a.w_tc = d.w_tc; a.cout_pad_tc = d.cout_pad_tc; a.bias = d.bias;
    a.up = e.arena ? Builder::ptr(e, p, up) : (const void*)16; a.up_ld = bu.ld; a.up_h = bu.h; a.up_w = bu.w;
    a.out = e.arena ? Builder::ptr(e, p, out) : (void*)16; a.out_ld = p.bufs[out].ld;
    a.N = bi.n; a.H = bi.h; a.W = bi.w; a.Cin = d.cin; a.K = d.cout;
    return a;
  };
  const bool ladder = exact2 && dtype == LEDB200_BF16 && e.cfg.conv_backend != 1 &&
                      ladder_eligible(rung_args(p, h + "head_x2", x2h, xc, hx2)) &&
                      ladder_eligible(rung_args(p, h + "head_x1", x1h, hx2, hx1)) &&
                      B.conv_uses_tc({e.conv_by_name.at(h + "conv_seg"), hf, xc});
  if (ladder) {
    p.bufs[xc].f16 = p.bufs[hx1].f16 = p.bufs[hx2].f16 = 1;
    // the rungs are stored as IEEE fp16 (same 2 bytes, 11-bit mantissa): tighter than bf16, and class logits are far
    // inside fp16's range (stores saturate at +-65504)
    B.conv(h + "conv_seg", hf, xc, -1, false, -1, -1, 0, 0, true);            // xc (fp16)
    auto add_rung = [&](const std::string& cname, int in, int up, int out, bool last) {
      const ConvDef& d = e.convs[e.conv_by_name.at(cname)];
      const Buf& bi = p.bufs[in];
      const double npo = (double)bi.n * bi.h * bi.w;
      p.ops.push_back({cname, [=](ledb200_handle& e, Plan& p, cudaStream_t st) -> int {
        LadderArgs a = rung_args(p, cname, in, up, out);
        if (last && !e.ext_logits) { a.final_argmax = 1; a.pred = e.ext_pred; a.pred_i64 = e.ext_pred_dtype == LEDB200_I64; }
        return launch_ladder(a, st);
      }, K_CONV_TC, 2.0 * npo * d.cout * d.cin * 9, 0.0});
      B.tag();
      // algorithmic bytes (SURVEY 8d): input once, the rung below once, weights; the rung written once - except for the
      // last rung on the label-only path, which writes 1 B per full-resolution pixel instead
      const Buf& bu = p.bufs[up];
      p.ops.back().bytes = 2.0 * (npo * d.cin + (double)bu.n * bu.h * bu.w * d.cout + (double)d.cout * d.cin * 9) +
                           (last ? 4.0 * npo : 2.0 * npo * d.cout);
    };
    add_rung(h + "head_x2", x2h, xc, hx2, false);      // hx2 buffer holds r2 (fp16)
    add_rung(h + "head_x1", x1h, hx2, hx1, true);      // labels, or r1 (fp16) when the logits are wanted
    p.ops.push_back({"tail.up2_argmax", [=](ledb200_handle& e, Plan& p, cudaStream_t st) -> int {
      if (!e.ext_logits) return LEDB200_OK;            // label-only path: head_x1 already wrote the labels
      Tail2Args a;
      const Buf& b1 = p.bufs[hx1];
      a.r1 = static_cast<const __half*>(Builder::ptr(e, p, hx1)); a.ld = b1.ld; a.N = b1.n; a.K = K; a.h2 = b1.h; a.w2 = b1.w;
      a.pred = e.ext_pred; a.pred_dtype = e.ext_pred_dtype; a.logits = e.ext_logits;
      return launch_tail2(a, st);
    }, K_TAIL, 0.0, 0.0});
    B.tag();
    return;
  }
  B.conv(h + "conv_seg", hf, xc);
  B.conv(h + "head_x1", x1h, hx1, -1, true);
  B.conv(h + "head_x2", x2h, hx2, -1, true);
  p.ops.push_back({"tail.fuse_argmax", [=](ledb200_handle& e, Plan& p, cudaStream_t st) -> int {
    TailArgs a;
    const Buf &bc = p.bufs[xc], &b2 = p.bufs[hx2], &b1 = p.bufs[hx1];
    a.xc = Builder::ptr(e, p, xc); a.hx2 = Builder::ptr(e, p, hx2); a.hx1 = Builder::ptr(e, p, hx1);
    a.xc_ld = bc.ld; a.hx2_ld = b2.ld; a.hx1_ld = b1.ld; a.dtype = dtype;
    a.N = bc.n; a.K = K; a.hc = bc.h; a.wc = bc.w; a.h4 = b2.h; a.w4 = b2.w; a.h2 = b1.h; a.w2 = b1.w;
    a.pred = e.ext_pred; a.pred_dtype = e.ext_pred_dtype; a.logits = e.ext_logits;
    return launch_tail(a, st);
  }, K_TAIL, 0.0, 0.0});
  B.tag();
  {
    const Buf &bc = p.bufs[xc], &b2 = p.bufs[hx2], &b1 = p.bufs[hx1];
    const double px = (double)n * (bc.h * bc.w + b2.h * b2.w + b1.h * b1.w);
    p.ops.back().bytes = esize(e) * px * K + (double)n * p.ho * p.wo;     // K-channel logits in, 1 B label out
    p.ops.back().flops = (double)n * p.ho * p.wo * K * 8.0;
  }
}

void add_export(Builder& B, const std::string& bufname, float* ledb200_handle::*dst) {
  Plan& p = B.p;
  const int id = p.by_name.at(bufname);
  const int dtype = B.dt;
  p.ops.push_back({"export." + bufname, [=](ledb200_handle& e, Plan& p, cudaStream_t st) -> int {
    const Buf& b = p.bufs[id];
    return launch_nhwc_to_nchw(Builder::ptr(e, p, id), dtype, e.*dst, b.n, b.c, b.h, b.w, b.ld, st);
  }, K_LAYOUT, 0.0, 0.0});
}

// Stand-alone LEDHead.forward on caller-provided NCHW fp32 features: the pre-activation BN+ReLU is
// the CUDA-core conv's prologue (the features come from outside, so no producer can apply it).
void build_head_standalone(Builder& B, int h8, int w8, int h2, int w2, int h4, int w4) {
  ledb200_handle& e = B.e;
  Plan& p = B.p;
  const int n = p.n, K = e.cfg.num_classes, HC = e.cfg.head_channels, C = e.cfg.channels;
  const int dtype = B.dt;
  const std::string h = "decode_head.";
  auto pre_conv = [&](const std::string& cname, const std::string& bn, const float* ledb200_handle::*src, int cin,
                      int H, int W, int out) {
    const int ci = e.conv_by_name.at(cname), ai = aff(e, bn);
    p.ops.push_back({cname, [=](ledb200_handle& e, Plan& p, cudaStream_t st) -> int {
      ConvArgs a = conv_args(e.convs[ci], n, H, W);
      const int64_t HW = (int64_t)H * W;
      a.in = e.*src; a.in_dtype = LEDB200_F32; a.in_sn = cin * HW; a.in_sc = HW; a.in_sh = W; a.in_sw = 1;
      a.pre_scale = e.affs[ai].scale; a.pre_shift = e.affs[ai].shift; a.pre_relu = 1;
      a.out = Builder::ptr(e, p, out); a.out_ld = p.bufs[out].ld; a.out_dtype = dtype; a.relu = 1;
      return launch_conv(a, 1, "engine", st);
    }, K_CONV_DIRECT, 0.0, 0.0});
  };
  const int hf = B.buf("head.feat", n, h8, w8, HC);
  pre_conv(h + "head", h + "head.0.bn", &ledb200_handle::in_c5, 4 * C, h8, w8, hf);
  const int xc = B.buf("xc", n, h8, w8, K, kpad(K));
  B.conv(h + "conv_seg", hf, xc);
  const int hx1 = B.buf("hx1", n, h2, w2, K, kpad(K));
  pre_conv(h + "head_x1", h + "head_x1.0.bn", &ledb200_handle::in_x1, C, h2, w2, hx1);
  const int hx2 = B.buf("hx2", n, h4, w4, K, kpad(K));
  pre_conv(h + "head_x2", h + "head_x2.0.bn", &ledb200_handle::in_x2, C, h4, w4, hx2);
  add_export(B, "xc", &ledb200_handle::ext_xc);
  add_export(B, "hx1", &ledb200_handle::ext_hx1);
  add_export(B, "hx2", &ledb200_handle::ext_hx2);
}

// Head + fused tail on caller-owned NHWC features in the engine's dtype (a trunk that is not the R0 plan, e.g.
// LEDNet(variant='led')): the three pre-activation BN + ReLU become one affine pass each, then the same fused head as
// the whole-inference plan (tensor-core ladder, labels without full-resolution logits).
void build_head_nhwc(Builder& B, int h8, int w8, int h2, int w2, int h4, int w4) {
  ledb200_handle& e = B.e;
  Plan& p = B.p;
  const int n = p.n, C = e.cfg.channels;
  const int dtype = B.dt;
  auto pre = [&](const std::string& name, const std::string& bn, const float* ledb200_handle::*src, int c, int H, int W) {
    const int out = B.buf(name, n, H, W, c);
    const int ai = aff(e, bn);
    p.ops.push_back({name + " (pre-activation)", [=](ledb200_handle& e, Plan& p, cudaStream_t st) -> int {
      AffineArgs a;
      a.in = e.*src; a.out_a = Builder::ptr(e, p, out); a.sa = e.affs[ai].scale; a.ba = e.affs[ai].shift;
      a.dtype = dtype; a.npix = (int64_t)n * H * W; a.C = c;
      return launch_affine_relu(a, st);
    }, K_AFFINE, 0.0, 2.0 * esize(e) * (double)n * H * W * c});
    B.tag();
  };
  pre("c5h", "decode_head.head.0.bn", &ledb200_handle::in_c5, 4 * C, h8, w8);
  pre("x1h", "decode_head.head_x1.0.bn", &ledb200_handle::in_x1, C, h2, w2);
  pre("x2h", "decode_head.head_x2.0.bn", &ledb200_handle::in_x2, C, h4, w4);
  build_head_fused(B);
}

void drop_graphs(ledb200_handle& e);

int get_plan(ledb200_handle& e, int kind, int n, int h, int w, int extra[6], Plan** out) {
  std::string key = std::to_string(kind) + ":" + std::to_string(n) + ":" + std::to_string(h) + ":" + std::to_string(w);
  if (extra) for (int i = 0; i < 6; ++i) key += ":" + std::to_string(extra[i]);
  auto it = e.plans.find(key);
  if (it == e.plans.end()) {
    auto p = std::make_unique<Plan>();
    p->kind = kind; p->n = n; p->h = h; p->w = w;
    Builder B(e, *p);
    try {
      if (kind == PLAN_INFER) { build_trunk(B, false, true); build_head_fused(B); }
      else if (kind == PLAN_BACKBONE) {
        build_trunk(B, true, false);
        add_export(B, "c5", &ledb200_handle::ext_c5);
        add_export(B, "x1", &ledb200_handle::ext_x1);
        add_export(B, "x2", &ledb200_handle::ext_x2);
      } else if (kind == PLAN_HEAD_NHWC) {
        build_head_nhwc(B, extra[0], extra[1], extra[2], extra[3], extra[4], extra[5]);
      } else {
        build_head_standalone(B, extra[0], extra[1], extra[2], extra[3], extra[4], extra[5]);
      }
    } catch (const std::exception& ex) {
      return fail(LEDB200_EINVAL, std::string("plan build failed: ") + ex.what());
    }
    it = e.plans.emplace(key, std::move(p)).first;
  }
  Plan* p = it->second.get();
  if (p->arena > e.arena_cap) {
    LEDB_CUDA_OK(cudaDeviceSynchronize());
    drop_graphs(e);
    if (e.arena) LEDB_CUDA_OK(cudaFree(e.arena));
    e.arena = nullptr; e.arena_cap = 0;
    void* q = nullptr;
    if (cudaMalloc(&q, p->arena) != cudaSuccess) {
      cudaGetLastError();
      return fail(LEDB200_ENOMEM, "cannot allocate " + std::to_string(p->arena >> 20) + " MiB activation workspace");
    }
    e.arena = (char*)q; e.arena_cap = p->arena;
    // debugging aid: fill the workspace with a NaN pattern so that any read of a never-written byte shows up
    if (const char* ps = getenv("LEDB200_POISON")) LEDB_CUDA_OK(cudaMemset(q, atoi(ps), p->arena));
  }
  *out = p;
  return LEDB200_OK;
}

void drop_graphs(ledb200_handle& e) {
  for (auto& kv : e.plans)
    for (auto& g : kv.second->graphs) if (g.exec) cudaGraphExecDestroy(g.exec);
  for (auto& kv : e.plans) kv.second->graphs.clear();
}

int ensure_streams(ledb200_handle& e) {
  if (e.cap[0]) return LEDB200_OK;
  for (int i = 0; i < 2; ++i) LEDB_CUDA_OK(cudaStreamCreateWithFlags(&e.cap[i], cudaStreamNonBlocking));
  LEDB_CUDA_OK(cudaEventCreateWithFlags(&e.ev_fork, cudaEventDisableTiming));
  LEDB_CUDA_OK(cudaEventCreateWithFlags(&e.ev_join, cudaEventDisableTiming));
  for (int i = 0; i < 2; ++i) LEDB_CUDA_OK(cudaEventCreateWithFlags(&e.ev_x[i], cudaEventDisableTiming));
  return LEDB200_OK;
}

// Issue every op of the plan on two streams: lane 0 = s0, lane 1 = s1.  s1 forks from s0 at the start
// and joins back at the end; an op flagged wait_other first makes its stream wait for the other
// stream's tail.  Works both eagerly and under stream capture (the events become graph edges).
int issue_ops(ledb200_handle& e, Plan& p, cudaStream_t s0, cudaStream_t s1) {
  const bool lanes = e.use_lanes && s1 != nullptr;
  cudaStream_t ss[2] = {s0, lanes ? s1 : s0};
  if (lanes) {
    LEDB_CUDA_OK(cudaEventRecord(e.ev_fork, s0));
    LEDB_CUDA_OK(cudaStreamWaitEvent(s1, e.ev_fork, 0));
  }
  for (auto& op : p.ops) {
    const int l = lanes ? op.lane : 0;
    if (lanes && op.wait_other) {
      LEDB_CUDA_OK(cudaEventRecord(e.ev_x[1 - l], ss[1 - l]));
      LEDB_CUDA_OK(cudaStreamWaitEvent(ss[l], e.ev_x[1 - l], 0));
    }
    int rc = op.fn(e, p, ss[l]);
    if (rc) { set_error("op '" + op.name + "': " + g_err); return rc; }
  }
  if (lanes) {
    LEDB_CUDA_OK(cudaEventRecord(e.ev_join, s1));
    LEDB_CUDA_OK(cudaStreamWaitEvent(s0, e.ev_join, 0));
  }
  return LEDB200_OK;
}

std::vector<const void*> ext_key(const ledb200_handle& e) {
  return {e.ext_img, (const void*)(intptr_t)e.ext_layout, e.ext_pred, (const void*)(intptr_t)e.ext_pred_dtype,
          e.ext_logits, e.ext_c5, e.ext_x1, e.ext_x2, e.in_c5, e.in_x1, e.in_x2, e.ext_xc, e.ext_hx1, e.ext_hx2,
          e.arena};
}

int run_plan(ledb200_handle& e, Plan& p, cudaStream_t st) {
  e.last_plan = &p;
  int rc = ensure_streams(e);
  if (rc) return rc;
  if (!e.use_graph) {
    // eager: lane 0 is the caller's stream, lane 1 the engine's side stream
    return issue_ops(e, p, st, e.cap[1]);
  }
  // one CUDA graph per (plan, caller buffers): kernel arguments, tensor maps and the two-lane
  // dependency structure are baked at capture; replay is a single launch on the caller's stream
  const std::vector<const void*> key = ext_key(e);
  for (auto& g : p.graphs)
    if (g.key == key) { LEDB_CUDA_OK(cudaGraphLaunch(g.exec, st)); return LEDB200_OK; }
  if (p.graphs.size() >= 8) {   // callers that allocate fresh outputs every call: keep the cache bounded
    if (p.graphs.front().exec) cudaGraphExecDestroy(p.graphs.front().exec);
    p.graphs.erase(p.graphs.begin());
  }
  LEDB_CUDA_OK(cudaStreamBeginCapture(e.cap[0], cudaStreamCaptureModeRelaxed));
  rc = issue_ops(e, p, e.cap[0], e.cap[1]);
  cudaGraph_t graph = nullptr;
  cudaError_t ce = cudaStreamEndCapture(e.cap[0], &graph);
  if (rc) { if (graph) cudaGraphDestroy(graph); cudaGetLastError(); return rc; }
  if (ce != cudaSuccess) { cudaGetLastError(); return fail(LEDB200_ECUDA, std::string("graph capture: ") + cudaGetErrorString(ce)); }
  GraphEntry ge; ge.key = key;
  ce = cudaGraphInstantiate(&ge.exec, graph, 0);
  cudaGraphDestroy(graph);
  if (ce != cudaSuccess) return fail(LEDB200_ECUDA, std::string("graph instantiate: ") + cudaGetErrorString(ce));
  p.graphs.push_back(ge);
  LEDB_CUDA_OK(cudaGraphLaunch(ge.exec, st));
  return LEDB200_OK;
}

int check_ready(ledb200_handle* h) {
  if (!h) return fail(LEDB200_EINVAL, "null handle");
  if (!h->finalized) return fail(LEDB200_ESTATE, "ledb200_finalize() has not been called");
  LEDB_CUDA_OK(cudaSetDevice(h->cfg.device));
  return LEDB200_OK;
}

}  // namespace
}  // namespace ledb

// ====================================================================== C ABI
extern "C" {

int ledb200_version(void) { return LEDB200_VERSION; }
const char* ledb200_last_error(void) { return g_err.c_str(); }

int ledb200_create(const ledb200_cfg* cfg, ledb200_handle** out) {
  if (!cfg || !out) return fail(LEDB200_EINVAL, "null argument");
  if (cfg->align_corners) return fail(LEDB200_EINVAL, "align_corners=True is not supported (config uses False)");
  if (cfg->dtype != LEDB200_F32 && cfg->dtype != LEDB200_BF16) return fail(LEDB200_EINVAL, "dtype must be F32 or BF16");
  if (cfg->variant != 0) return fail(LEDB200_EINVAL, "only variant 0 (R0 trunk) exists");
  if (cfg->in_channels != 3) return fail(LEDB200_EINVAL, "in_channels must be 3");
  if (cfg->channels < 8 || cfg->channels % 8 || cfg->ppm_channels % 8 || cfg->head_channels % 8)
    return fail(LEDB200_EINVAL, "channels, ppm_channels and head_channels must be multiples of 8");
  if (cfg->num_classes < 2 || cfg->num_classes > 255) return fail(LEDB200_EINVAL, "num_classes must be in [2,255]");
  int ndev = 0;
  LEDB_CUDA_OK(cudaGetDeviceCount(&ndev));
  if (cfg->device < 0 || cfg->device >= ndev) return fail(LEDB200_EINVAL, "bad device ordinal");
  auto* h = new (std::nothrow) ledb200_handle();
  if (!h) return fail(LEDB200_ENOMEM, "out of host memory");
  h->cfg = *cfg;
  h->use_graph = getenv("LEDB200_NO_GRAPH") ? 0 : 1;
  h->use_lanes = getenv("LEDB200_NO_LANES") ? 0 : 1;
  try { define_model(*h); } catch (const std::exception& ex) { delete h; return fail(LEDB200_EINVAL, ex.what()); }
  *out = h;
  return LEDB200_OK;
}

int ledb200_destroy(ledb200_handle* h) {
  if (!h) return LEDB200_OK;
  cudaSetDevice(h->cfg.device);
  cudaDeviceSynchronize();
  drop_graphs(*h);
  for (int i = 0; i < 2; ++i) { if (h->cap[i]) cudaStreamDestroy(h->cap[i]); if (h->ev_x[i]) cudaEventDestroy(h->ev_x[i]); }
  if (h->ev_fork) cudaEventDestroy(h->ev_fork);
  if (h->ev_join) cudaEventDestroy(h->ev_join);
  for (auto& d : h->convs) free_conv(d);
  for (void* p : h->dev_allocs) cudaFree(p);
  if (h->arena) cudaFree(h->arena);
  delete h;
  return LEDB200_OK;
}

int ledb200_set_param(ledb200_handle* h, const char* name, const void* data, const int64_t* shape, int32_t ndim,
                      int32_t dtype) {
  if (!h || !name || !data || ndim < 0 || (ndim > 0 && !shape)) return fail(LEDB200_EINVAL, "null argument");
  if (h->finalized) return fail(LEDB200_ESTATE, "handle already finalized");
  const std::string k(name);
  if (k.size() > 20 && k.compare(k.size() - 19, 19, "num_batches_tracked") == 0) return LEDB200_OK;
  if (dtype != LEDB200_F32) return fail(LEDB200_EINVAL, k + ": parameters must be fp32");
  if (std::find(h->expected.begin(), h->expected.end(), k) == h->expected.end())
    return fail(LEDB200_ENOTFOUND, "unexpected parameter name: " + k);
  int64_t n = 1;
  HostTensor t;
  for (int i = 0; i < ndim; ++i) { n *= shape[i]; t.shape.push_back(shape[i]); }
  t.v.assign((const float*)data, (const float*)data + n);
  h->params[k] = std::move(t);
  return LEDB200_OK;
}

int ledb200_num_params(ledb200_handle* h) { return h ? (int)h->expected.size() : 0; }
const char* ledb200_param_name(ledb200_handle* h, int32_t i) {
  if (!h || i < 0 || i >= (int)h->expected.size()) return nullptr;
  return h->expected[i].c_str();
}

int ledb200_finalize(ledb200_handle* h) {
  if (!h) return fail(LEDB200_EINVAL, "null handle");
  if (h->finalized) return LEDB200_OK;
  LEDB_CUDA_OK(cudaSetDevice(h->cfg.device));
  return finalize(*h);
}

int ledb200_forward_infer(ledb200_handle* h, const void* img, int32_t img_layout, int32_t N, int32_t H, int32_t W,
                          void* pred, int32_t pred_dtype, float* logits_opt, void* stream) {
  int rc = check_ready(h);
  if (rc) return rc;
  if (!img || !pred) return fail(LEDB200_EINVAL, "null image or prediction buffer");
  if (N < 1 || H < 8 || W < 8) return fail(LEDB200_EINVAL, "need N >= 1 and H, W >= 8");
  if (img_layout < 0 || img_layout > 2) return fail(LEDB200_EINVAL, "bad image layout");
  if (pred_dtype != LEDB200_U8 && pred_dtype != LEDB200_I64) return fail(LEDB200_EINVAL, "pred dtype must be U8 or I64");
  Plan* p = nullptr;
  if ((rc = get_plan(*h, PLAN_INFER, N, H, W, nullptr, &p))) return rc;
  h->ext_img = img; h->ext_layout = img_layout; h->ext_pred = pred; h->ext_pred_dtype = pred_dtype;
  h->ext_logits = logits_opt;
  return run_plan(*h, *p, (cudaStream_t)stream);
}

int ledb200_backbone_forward(ledb200_handle* h, const void* img, int32_t img_layout, int32_t N, int32_t H, int32_t W,
                             float* c5, float* x1, float* x2, void* stream) {
  int rc = check_ready(h);
  if (rc) return rc;
  if (!img || !c5 || !x1 || !x2) return fail(LEDB200_EINVAL, "null buffer");
  if (N < 1 || H < 8 || W < 8) return fail(LEDB200_EINVAL, "need N >= 1 and H, W >= 8");
  Plan* p = nullptr;
  if ((rc = get_plan(*h, PLAN_BACKBONE, N, H, W, nullptr, &p))) return rc;
  h->ext_img = img; h->ext_layout = img_layout; h->ext_c5 = c5; h->ext_x1 = x1; h->ext_x2 = x2;
  return run_plan(*h, *p, (cudaStream_t)stream);
}

int ledb200_head_forward(ledb200_handle* h, const float* c5, const float* x1, const float* x2, int32_t N, int32_t h8,
                         int32_t w8, int32_t h2, int32_t w2, int32_t h4, int32_t w4, float* xc, float* hx1, float* hx2,
                         void* stream) {
  int rc = check_ready(h);
  if (rc) return rc;
  if (!c5 || !x1 || !x2 || !xc || !hx1 || !hx2) return fail(LEDB200_EINVAL, "null buffer");
  int extra[6] = {h8, w8, h2, w2, h4, w4};
  for (int v : extra) if (v < 1) return fail(LEDB200_EINVAL, "empty feature map");
  Plan* p = nullptr;
  if ((rc = get_plan(*h, PLAN_HEAD, N, 0, 0, extra, &p))) return rc;
  h->in_c5 = c5; h->in_x1 = x1; h->in_x2 = x2; h->ext_xc = xc; h->ext_hx1 = hx1; h->ext_hx2 = hx2;
  return run_plan(*h, *p, (cudaStream_t)stream);
}

int ledb200_head_infer(ledb200_handle* h, const void* c5, const void* x1, const void* x2, int32_t N, int32_t h8, int32_t w8,
                       int32_t h2, int32_t w2, int32_t h4, int32_t w4, void* pred, int32_t pred_dtype, float* logits_opt,
                       void* stream) {
  int rc = check_ready(h);
  if (rc) return rc;
  if (!c5 || !x1 || !x2 || !pred) return fail(LEDB200_EINVAL, "null buffer");
  if (pred_dtype != LEDB200_U8 && pred_dtype != LEDB200_I64) return fail(LEDB200_EINVAL, "pred dtype must be U8 or I64");
  int extra[6] = {h8, w8, h2, w2, h4, w4};
  for (int v : extra) if (v < 1) return fail(LEDB200_EINVAL, "empty feature map");
  if (N < 1) return fail(LEDB200_EINVAL, "need N >= 1");
  Plan* p = nullptr;
  if ((rc = get_plan(*h, PLAN_HEAD_NHWC, N, 0, 0, extra, &p))) return rc;
  h->in_c5 = (const float*)c5; h->in_x1 = (const float*)x1; h->in_x2 = (const float*)x2;
  h->ext_pred = pred; h->ext_pred_dtype = pred_dtype; h->ext_logits = logits_opt;
  return run_plan(*h, *p, (cudaStream_t)stream);
}

int ledb200_debug_fetch(ledb200_handle* h, const char* buffer_name, float* host_out, int64_t capacity, int32_t* shape4,
                        void* stream) {
  int rc = check_ready(h);
  if (rc) return rc;
  if (!h->last_plan) return fail(LEDB200_ESTATE, "no forward has run yet");
  Plan& p = *h->last_plan;
  auto it = p.by_name.find(buffer_name ? buffer_name : "");
  if (it == p.by_name.end()) return fail(LEDB200_ENOTFOUND, std::string("no buffer named ") + (buffer_name ? buffer_name : "(null)"));
  const Buf& b = p.bufs[it->second];
  const int64_t n = (int64_t)b.n * b.c * b.h * b.w;
  if (shape4) { shape4[0] = b.n; shape4[1] = b.c; shape4[2] = b.h; shape4[3] = b.w; }
  if (!host_out || capacity < n) return fail(LEDB200_EINVAL, "host buffer too small: need " + std::to_string(n));
  float* tmp = nullptr;
  LEDB_CUDA_OK(cudaMalloc(&tmp, n * sizeof(float)));
  cudaStream_t st = (cudaStream_t)stream;
  rc = launch_nhwc_to_nchw(h->arena + b.off, b.f16 ? 5 /* fp16 */ : h->cfg.dtype, tmp, b.n, b.c, b.h, b.w, b.ld, st);
  if (!rc) {
    cudaError_t ce = cudaMemcpyAsync(host_out, tmp, n * sizeof(float), cudaMemcpyDeviceToHost, st);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(st);
    if (ce != cudaSuccess) rc = fail(LEDB200_ECUDA, cudaGetErrorString(ce));
  }
  cudaFree(tmp);
  return rc;
}

int ledb200_plan_launches(ledb200_handle* h) { return (h && h->last_plan) ? (int)h->last_plan->ops.size() : 0; }
const char* ledb200_op_name(ledb200_handle* h, int32_t i) {
  if (!h || !h->last_plan || i < 0 || i >= (int)h->last_plan->ops.size()) return nullptr;
  return h->last_plan->ops[i].name.c_str();
}

int ledb200_op_info(ledb200_handle* h, int32_t i, double* out3) {
  if (!h || !h->last_plan || !out3 || i < 0 || i >= (int)h->last_plan->ops.size())
    return fail(LEDB200_EINVAL, "op_info: bad index or no plan");
  const Op& o = h->last_plan->ops[i];
  out3[0] = o.flops; out3[1] = o.bytes; out3[2] = (double)o.kind;
  return LEDB200_OK;
}

int ledb200_profile_ops(ledb200_handle* h, int32_t iters, float* ms_out, int32_t cap, void* stream) {
  int rc = check_ready(h);
  if (rc) return rc;
  if (!h->last_plan) return fail(LEDB200_ESTATE, "no forward has run yet");
  Plan& p = *h->last_plan;
  cudaStream_t st = (cudaStream_t)stream;
  cudaEvent_t e0, e1;
  LEDB_CUDA_OK(cudaEventCreate(&e0));
  LEDB_CUDA_OK(cudaEventCreate(&e1));
  if (iters < 1) iters = 1;
  for (int i = 0; i < (int)p.ops.size(); ++i) {
    if ((rc = p.ops[i].fn(*h, p, st))) break;   // warm
    cudaEventRecord(e0, st);
    for (int k = 0; k < iters && !rc; ++k) rc = p.ops[i].fn(*h, p, st);
    cudaEventRecord(e1, st);
    if (rc) break;
    if (cudaEventSynchronize(e1) != cudaSuccess) { rc = fail(LEDB200_ECUDA, "event sync failed"); break; }
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    if (i < cap && ms_out) ms_out[i] = ms / iters;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  return rc ? rc : (int)p.ops.size();
}

}  // extern "C"
