// MiT-EVP encoder + SegFormer embedding head: weight packing and the forward schedule.
//
// replaces MixVisionTransformerEVP.forward(x, y, flow, return_features=True) (mix_transformer_evp.py:418-449):
// forward_features (:352-416), PromptGenerator.init_prompts / init_prompt / get_prompt (:718-815), Block (:167-171),
// Attention (:110-131), Mlp + DWConv (:60-67, :24-30), OverlapPatchEmbed (:209-215), OpticalFlowEncoder (:838-859),
// MotionGuidedCrossAttention (:878-890) and SegFormerHead.forward (segformer_head.py:137-173).
//
// Data layout in HBM: every activation is token-major == NHWC ([frames*H*W, C]); the residual stream is fp32,
// every GEMM operand is bf16, accumulation fp32.  A forward is a static list of kernel launches ("plan") built once
// per (micro-batch, H, W, workspace) and replayed; frames are processed in micro-batches so the working set stays
// in the 126 MB L2.
#include <math.h>
#include <stdio.h>
#include <string.h>

#include <map>
#include <memory>
#include <utility>
#include <string>
#include <type_traits>
#include <variant>
#include <vector>

#include "gemm.cuh"
#include "host.cuh"
#include "kernels.cuh"

namespace sv {
namespace {

struct Lin {        // packed nn.Linear / patchified conv: bf16 W[N, ldw] + fp32 bias[N]
  size_t w = 0;     // element offset into the bf16 blob
  size_t b = 0;     // element offset into the fp32 blob
  int N = 0, K = 0, ldw = 0;
  bool has_bias = true;
};
struct Norm {       // LayerNorm affine, fp32
  size_t g = 0, b = 0;
  int C = 0;
};
struct BlockW {
  Norm n1, n2, srn;
  Lin q, kv, proj, sr, fc1, fc2;
  Lin fc2cat;  // [fc2 | shared_mlp] along K: x += fc2(h) + shared_mlp(T_next) in one GEMM (blocks that have a successor)
  size_t dw_w = 0, dw_b = 0;  // fp32 [9][4C], [4C]
};
struct StageW {
  Lin pe, emb, shared, hc;
  Norm pe_norm, hc_norm, norm;
  Lin lw_all;  // all lightweight_mlp{s}_{i} of the stage stacked along N: T_all = GELU(P . lw_all^T) in ONE GEMM (P does not depend on the block)
  std::vector<BlockW> blk;
};
struct CrossW {
  Lin q, kv, out;
  Norm norm;
};

// profile classes (sv_evp_get_profile, the `kind` column of sv_evp_dump_profile); the order is part of the ABI
enum OpKind { OP_GEMM, OP_LN, OP_IM2COL, OP_DWCONV, OP_ATTN, OP_GAUSS, OP_BILINEAR, OP_MEAN, OP_STEM, OP_KINDS };

// The pointers of one forward call for one micro-batch: a plan is built once and replayed on every call's inputs and outputs.
struct CallIO {
  const float *x, *seg, *flow; float* out;
  float* const* maps;  // per encoder block, where this micro-batch's attention maps go (capture plans only)
  float* const* stage_out;  // per stage, where this micro-batch's fp32 NCHW stage map goes (encoder-only plans only)
};
// where im2col and the stem read their fp32 NCHW input: a workspace buffer, or the call's x or flow
enum Ext { EXT_NONE, EXT_X, EXT_FLOW };
const float* nchw_input(Ext ext, const float* ws, const CallIO& io) { return ext == EXT_X ? io.x : ext == EXT_FLOW ? io.flow : ws; }
struct ProfCols { long long M; int i[5]; };  // columns M, i0..i4 of a non-GEMM row of sv_evp_dump_profile

// One record per launch form: its launcher's arguments under the launcher's names and in its order, and its profile class.
struct GemmOp {  // GEMM or implicit-GEMM conv
  static constexpr OpKind kind = OP_GEMM;
  GemmPlan plan;
  int launch(const CallIO&, cudaStream_t st) const { return gemm_launch(plan, st); }
};
struct LayerNormOp {  // out_patch: optional second bf16 copy in the sr conv's patch order (pH x pW grid, psr x psr patches)
  static constexpr OpKind kind = OP_LN;
  const float *x, *gamma, *beta; float eps; int64_t rows; int C; float* out_f32; bf16 *out_bf16, *out_patch; int pH, pW, psr;
  int launch(const CallIO&, cudaStream_t st) const { return launch_layernorm_patch(x, gamma, beta, eps, rows, C, out_f32, out_bf16, out_patch, pH, pW, psr, st); }
  ProfCols cols() const { return {rows, {C, pH, pW, psr, 0}}; }
};
struct Im2colOp {
  static constexpr OpKind kind = OP_IM2COL;
  Ext ext; const float* src_nchw_f32; const bf16* src_nhwc_bf16; int B, Cin, H, W, k, stride, pad; bf16* out; int64_t ldo;
  int launch(const CallIO& io, cudaStream_t st) const {
    return launch_im2col(nchw_input(ext, src_nchw_f32, io), src_nhwc_bf16, B, Cin, H, W, k, stride, pad, out, ldo, st);
  }
  ProfCols cols() const { return {ldo, {B, Cin, H, W, k}}; }
};
struct DwconvTmaOp {
  static constexpr OpKind kind = OP_DWCONV;
  DwconvPlan plan;
  int launch(const CallIO&, cudaStream_t st) const { return dwconv_tma_launch(plan, st); }
  ProfCols cols() const { return {plan.ldo, {plan.B, plan.H, plan.W, plan.C, 0}}; }
};
struct DwconvOp {  // channel counts the TMA form does not take (dwconv_tma_supported)
  static constexpr OpKind kind = OP_DWCONV;
  const bf16* x; const float *w9c, *bias; int B, H, W, C; bf16* out; int64_t ldo;
  int launch(const CallIO&, cudaStream_t st) const { return launch_dwconv3x3_gelu(x, w9c, bias, B, H, W, C, out, ldo, st); }
  ProfCols cols() const { return {ldo, {B, H, W, C, 0}}; }
};
struct AttnTcOp {
  static constexpr OpKind kind = OP_ATTN;
  AttnTcPlan plan;
  int64_t ldq; int hd;  // for the profile only: the plan keeps neither
  int launch(const CallIO&, cudaStream_t st) const { return attention_tc_launch(plan, st); }
  ProfCols cols() const { return {ldq, {plan.B, plan.heads, plan.Nq, plan.Nkv, hd}}; }
};
struct AttnOp {  // mma.sync kernels: head_dim 20/32/40, or SURGVID_ATTN_TC=0
  static constexpr OpKind kind = OP_ATTN;
  const bf16* q; int64_t ldq; const bf16* k; int64_t ldk; const bf16* v; int64_t ldv; bf16* o; int64_t ldo; int B, heads, Nq, Nkv, hd; float scale;
  int launch(const CallIO&, cudaStream_t st) const { return launch_attention(q, ldq, k, ldk, v, ldv, o, ldo, B, heads, Nq, Nkv, hd, scale, st); }
  ProfCols cols() const { return {ldq, {B, heads, Nq, Nkv, hd}}; }
};
struct ProbsOp {  // softmax(Q K^T * scale) of encoder block `block` into the call's maps[block]
  static constexpr OpKind kind = OP_ATTN;
  const bf16* q; int64_t ldq; const bf16* k; int64_t ldk; int B, heads, Nq, Nkv, hd; float scale; int block;
  int launch(const CallIO& io, cudaStream_t st) const { return launch_attention_probs(q, ldq, k, ldk, B, heads, Nq, Nkv, hd, scale, io.maps[block], st); }
  ProfCols cols() const { return {ldq, {B, heads, Nq, Nkv, hd}}; }
};
struct StageNormOp {  // stage norm of the encoder-only plans: fp32 result channel-major into the call's stage_out[stage]
  static constexpr OpKind kind = OP_LN;
  const float *x, *gamma, *beta; float eps; int64_t rows; int C, tokens; bf16* out_bf16; int stage;
  int launch(const CallIO& io, cudaStream_t st) const {
    return launch_layernorm_nchw(x, gamma, beta, eps, rows, C, tokens, io.stage_out[stage], out_bf16, st);
  }
  ProfCols cols() const { return {rows, {C, tokens, 0, 0, stage}}; }
};
struct GaussOp {  // of the call's seg
  static constexpr OpKind kind = OP_GAUSS;
  float* out; int planes, H, W;
  int launch(const CallIO& io, cudaStream_t st) const { return launch_gauss5x5(io.seg, out, planes, H, W, st); }
  ProfCols cols() const { return {0, {planes, H, W, 0, 0}}; }
};
struct BilinearOp {
  static constexpr OpKind kind = OP_BILINEAR;
  const bf16* x; int B, H, W, C, Ho, Wo; bf16* out; int64_t ldo;
  int launch(const CallIO&, cudaStream_t st) const { return launch_bilinear_tokens(x, B, H, W, C, Ho, Wo, out, ldo, st); }
  ProfCols cols() const { return {ldo, {B, H, W, C, Ho}}; }
};
struct MeanOp {  // into the call's out
  static constexpr OpKind kind = OP_MEAN;
  const float* x; int B, tokens, C;
  int launch(const CallIO& io, cudaStream_t st) const { return launch_token_mean(x, B, tokens, C, io.out, st); }
  ProfCols cols() const { return {0, {B, tokens, C, 0, 0}}; }
};
struct StemOp {  // mode 0: LayerNorm, 1: ReLU
  static constexpr OpKind kind = OP_STEM;
  Ext ext; const float* src; const bf16* w; int ldw; const float *bias, *gamma, *beta; float eps; int mode; int B, Cin, H, W, Cout;
  float* out_f32; bf16* out_bf16;
  int launch(const CallIO& io, cudaStream_t st) const {
    return launch_stem_conv(nchw_input(ext, src, io), w, ldw, bias, gamma, beta, eps, mode, B, Cin, H, W, Cout, out_f32, out_bf16, st);
  }
  ProfCols cols() const { return {0, {B, Cin, H, W, Cout}}; }
};

struct Op {
  std::variant<GemmOp, LayerNormOp, Im2colOp, DwconvTmaOp, DwconvOp, AttnTcOp, AttnOp, ProbsOp, StageNormOp, GaussOp, BilinearOp, MeanOp, StemOp>
      rec;
  double alg_bytes = 0.0;         // algorithmic HBM bytes of this launch (operands + results once)
  mutable double prof_ms = 0.0;   // filled only in profiling mode
  mutable long long prof_n = 0;
  OpKind kind() const { return std::visit([](const auto& r) { return r.kind; }, rec); }
};

struct Tap {
  const bf16* ptr;
  int64_t elems;
};

struct Plan {
  int n = 0, H = 0, W = 0;
  bool with_flow = false;
  void* ws = nullptr;
  size_t need = 0;        // workspace bytes this plan addresses
  uint64_t last_use = 0;  // for eviction
  std::vector<Op> ops;
  std::map<std::string, Tap> taps;
  double gemm_flops = 0.0;
  double bytes_by_kind[OP_KINDS] = {};
};

// bump allocator over the caller's workspace (dry run when base == nullptr)
struct Arena {
  char* base;
  size_t off = 0;
  std::vector<std::pair<size_t, size_t>> allocs;   // (offset, bytes) of every buffer handed out, for the bounds check of the plan
  explicit Arena(void* b) : base(static_cast<char*>(b)) {}
  template <typename T>
  T* get(size_t count) {
    off = (off + 255) & ~static_cast<size_t>(255);
    T* p = reinterpret_cast<T*>(base + off);
    allocs.emplace_back(off, count * sizeof(T));
    off += count * sizeof(T);
    return p;
  }
  // does [p, p + bytes) lie inside ONE buffer of the arena?  (a launch that runs past its buffer into a neighbour corrupts silently)
  bool contains(const void* p, size_t bytes) const {
    const size_t o = static_cast<size_t>(static_cast<const char*>(p) - base);
    for (const auto& a : allocs)
      if (o >= a.first && o + bytes <= a.first + a.second) return true;
    return false;
  }
};

constexpr size_t kMaxPlans = 16;  // distinct (micro-batch, H, W, flow) schedules kept per handle

struct StageGeom {
  int H, W, N, C, heads, sr, Hk, Wk, Nkv, hidden, Cp;
};

}  // namespace
}  // namespace sv

struct sv_evp {
  sv_evp_cfg cfg;
  int device = 0;
  sv::StateDict sd;
  sv::bf16* d_wb = nullptr;
  float* d_wf = nullptr;
  sv::StageW st[4];
  sv::Lin flow[4];
  sv::CrossW xa[2];
  sv::Lin head_c[4];   // index 0..3 = linear_c1..c4
  sv::Lin head_fuse;   // [E, 4E] (BN scale folded), bias = BN shift
  sv::Lin head_fold;   // [E, sum C_i] when cfg.fold_head
  size_t fc_w[2][2] = {{0, 0}, {0, 0}}, fc_b[2][2] = {{0, 0}, {0, 0}};  // fp32 classifier heads: [fc|fc_ant][layer]
  std::map<long long, std::unique_ptr<sv::Plan>> plans;  // bounded: see kMaxPlans
  uint64_t plan_clock = 0;
  sv::Plan* last_plan = nullptr;
  int64_t launches = 0;
  // optional per-kernel-class timing (CUDA events around every launch; bench.py's roofline pass)
  bool profile = false;
  double prof_ms[sv::OP_KINDS] = {};
  int64_t prof_n[sv::OP_KINDS] = {};
  double prof_gemm_flops = 0.0;
  double prof_bytes[sv::OP_KINDS] = {};
  std::vector<cudaEvent_t> prof_events;
};

namespace sv {
namespace {

// --------------------------------------------------------------------------------------------- packing
struct Packer {
  sv_evp* h;
  std::vector<uint16_t> wb;  // bf16 bits
  std::vector<float> wf;
  std::string err;

  static uint16_t to_bf16(float f) {  // round-to-nearest-even, as __float2bfloat16_rn
    uint32_t u;
    memcpy(&u, &f, 4);
    if ((u & 0x7fffffffu) > 0x7f800000u) return static_cast<uint16_t>((u >> 16) | 0x40);
    u += 0x7fffu + ((u >> 16) & 1u);
    return static_cast<uint16_t>(u >> 16);
  }
  size_t alloc_b(size_t n) { size_t o = wb.size(); wb.resize(o + ((n + 7) / 8) * 8, 0); return o; }
  size_t alloc_f(size_t n) { size_t o = wf.size(); wf.resize(o + ((n + 3) / 4) * 4, 0.f); return o; }

  const HostTensor* get(const std::string& key, const std::vector<int64_t>& shape) {
    const HostTensor* t;
    if (h->sd.get(key, shape, "evp pack_weights", &t) != SV_OK && err.empty()) err = sv_last_error();
    return t;
  }
  size_t vec(const std::string& key, int64_t n) {
    const HostTensor* t = get(key, {n});
    size_t o = alloc_f(n);
    if (t) std::copy(t->data.begin(), t->data.end(), wf.begin() + o);
    return o;
  }
  Norm norm(const std::string& p, int C) {
    Norm n;
    n.C = C;
    n.g = vec(p + ".weight", C);
    n.b = vec(p + ".bias", C);
    return n;
  }
  // nn.Linear weight [N, K]; optional per-row scale (BN fold)
  Lin linear_raw(const float* w, const float* bias, int N, int K, const float* row_scale = nullptr) {
    Lin l;
    l.N = N; l.K = K; l.ldw = round_up(K, 8);
    l.w = alloc_b(static_cast<size_t>(N) * l.ldw);
    for (int n = 0; n < N; ++n)
      for (int k = 0; k < K; ++k) wb[l.w + static_cast<size_t>(n) * l.ldw + k] = to_bf16(w[static_cast<size_t>(n) * K + k] * (row_scale ? row_scale[n] : 1.f));
    l.b = alloc_f(N);
    l.has_bias = bias != nullptr;
    if (bias) std::copy(bias, bias + N, wf.begin() + l.b);
    return l;
  }
  Lin linear(const std::string& p, int N, int K) {
    const HostTensor* w = get(p + ".weight", {N, K});
    const HostTensor* b = get(p + ".bias", {N});
    if (!w || !b) return Lin();
    return linear_raw(w->data.data(), b->data.data(), N, K);
  }
  // Conv2d weight [Cout, Cin, k, k] -> implicit-GEMM form [Cout, (kh, kw, cin)], optional BN fold
  Lin conv(const std::string& p, int Cout, int Cin, int k, const float* scale = nullptr, const float* shift = nullptr) {
    const HostTensor* w = get(p + ".weight", {Cout, Cin, k, k});
    const HostTensor* b = get(p + ".bias", {Cout});
    if (!w || !b) return Lin();
    const int K = k * k * Cin;
    std::vector<float> r(static_cast<size_t>(Cout) * K), bb(Cout);
    for (int co = 0; co < Cout; ++co) {
      for (int ci = 0; ci < Cin; ++ci)
        for (int kh = 0; kh < k; ++kh)
          for (int kw = 0; kw < k; ++kw)
            r[static_cast<size_t>(co) * K + (kh * k + kw) * Cin + ci] = w->data[((static_cast<size_t>(co) * Cin + ci) * k + kh) * k + kw];
      bb[co] = scale ? b->data[co] * scale[co] + shift[co] : b->data[co];
    }
    return linear_raw(r.data(), bb.data(), Cout, K, scale);
  }
  // BatchNorm2d (eval): scale = g / sqrt(var + 1e-5), shift = b - mean * scale
  bool bn(const std::string& p, int C, std::vector<float>* scale, std::vector<float>* shift) {
    const HostTensor* g = get(p + ".weight", {C});
    const HostTensor* b = get(p + ".bias", {C});
    const HostTensor* m = get(p + ".running_mean", {C});
    const HostTensor* v = get(p + ".running_var", {C});
    if (!g || !b || !m || !v) return false;
    scale->resize(C);
    shift->resize(C);
    for (int c = 0; c < C; ++c) {
      const double s = static_cast<double>(g->data[c]) / sqrt(static_cast<double>(v->data[c]) + 1e-5);
      (*scale)[c] = static_cast<float>(s);
      (*shift)[c] = static_cast<float>(static_cast<double>(b->data[c]) - static_cast<double>(m->data[c]) * s);
    }
    return true;
  }
};

int pack_all(sv_evp* h) {
  const sv_evp_cfg& c = h->cfg;
  Packer P;
  P.h = h;
  const int E = c.embedding_dim;
  const int ks[4] = {7, 3, 3, 3};
  for (int s = 0; s < 4; ++s) {
    const int C = c.embed_dims[s], Cp = C / 4, hid = C * c.mlp_ratio, sr = c.sr_ratios[s];
    const int cin = s == 0 ? 3 : c.embed_dims[s - 1];
    const int cinp = s == 0 ? 3 : c.embed_dims[s - 1] / 4;
    StageW& S = h->st[s];
    const std::string sn = std::to_string(s + 1);
    S.pe = P.conv("patch_embed" + sn + ".proj", C, cin, ks[s]);
    S.pe_norm = P.norm("patch_embed" + sn + ".norm", C);
    S.hc = P.conv("prompt_generator.handcrafted_generator" + sn + ".proj", Cp, cinp, ks[s]);
    S.hc_norm = P.norm("prompt_generator.handcrafted_generator" + sn + ".norm", Cp);
    S.emb = P.linear("prompt_generator.embedding_generator" + sn, Cp, C);
    S.shared = P.linear("prompt_generator.shared_mlp" + sn, C, Cp);
    S.blk.clear();
    for (int i = 0; i < c.depths[s]; ++i) {
      const std::string bp = "block" + sn + "." + std::to_string(i);
      BlockW B;
      B.n1 = P.norm(bp + ".norm1", C);
      B.q = P.linear(bp + ".attn.q", C, C);
      B.kv = P.linear(bp + ".attn.kv", 2 * C, C);
      B.proj = P.linear(bp + ".attn.proj", C, C);
      if (sr > 1) {
        B.sr = P.conv(bp + ".attn.sr", C, C, sr);
        B.srn = P.norm(bp + ".attn.norm", C);
      }
      B.n2 = P.norm(bp + ".norm2", C);
      B.fc1 = P.linear(bp + ".mlp.fc1", hid, C);
      B.fc2 = P.linear(bp + ".mlp.fc2", C, hid);
      const HostTensor* dw = P.get(bp + ".mlp.dwconv.dwconv.weight", {hid, 1, 3, 3});
      B.dw_w = P.alloc_f(static_cast<size_t>(9) * hid);
      if (dw)
        for (int ch = 0; ch < hid; ++ch)
          for (int t = 0; t < 9; ++t) P.wf[B.dw_w + static_cast<size_t>(t) * hid + ch] = dw->data[static_cast<size_t>(ch) * 9 + t];
      B.dw_b = P.vec(bp + ".mlp.dwconv.dwconv.bias", hid);
      S.blk.push_back(B);
    }
    {  // stacked lightweight MLPs: rows [i*Cp, (i+1)*Cp) = lightweight_mlp{s}_{i}.0
      std::vector<float> wa(static_cast<size_t>(c.depths[s]) * Cp * Cp, 0.f), ba(static_cast<size_t>(c.depths[s]) * Cp, 0.f);
      bool ok = true;
      for (int i = 0; i < c.depths[s]; ++i) {
        const std::string ln = "prompt_generator.lightweight_mlp" + sn + "_" + std::to_string(i) + ".0";
        const HostTensor* w = P.get(ln + ".weight", {Cp, Cp});
        const HostTensor* bb = P.get(ln + ".bias", {Cp});
        if (!w || !bb) { ok = false; break; }
        std::copy(w->data.begin(), w->data.end(), wa.begin() + static_cast<size_t>(i) * Cp * Cp);
        std::copy(bb->data.begin(), bb->data.end(), ba.begin() + static_cast<size_t>(i) * Cp);
      }
      if (ok) S.lw_all = P.linear_raw(wa.data(), ba.data(), c.depths[s] * Cp, Cp);
    }
    // Adapter fusion: the adapter term of block i+1, shared_mlp(GELU(lightweight_mlp_{i+1}(P))), does not depend on x, so it
    // is added by block i's fc2 GEMM: K-concatenated weight [W_fc2_i | W_shared], bias b_fc2_i + b_shared.
    {
      const HostTensor* wsh = P.get("prompt_generator.shared_mlp" + sn + ".weight", {C, Cp});
      const HostTensor* bsh = P.get("prompt_generator.shared_mlp" + sn + ".bias", {C});
      for (int i = 0; i + 1 < c.depths[s] && wsh && bsh; ++i) {
        const std::string bp = "block" + sn + "." + std::to_string(i);
        const HostTensor* w2 = P.get(bp + ".mlp.fc2.weight", {C, hid});
        const HostTensor* b2 = P.get(bp + ".mlp.fc2.bias", {C});
        if (!w2 || !b2) break;
        std::vector<float> wc(static_cast<size_t>(C) * (hid + Cp)), bc(C);
        for (int n = 0; n < C; ++n) {
          std::copy(w2->data.begin() + static_cast<size_t>(n) * hid, w2->data.begin() + static_cast<size_t>(n + 1) * hid, wc.begin() + static_cast<size_t>(n) * (hid + Cp));
          std::copy(wsh->data.begin() + static_cast<size_t>(n) * Cp, wsh->data.begin() + static_cast<size_t>(n + 1) * Cp,
                    wc.begin() + static_cast<size_t>(n) * (hid + Cp) + hid);
          bc[n] = b2->data[n] + bsh->data[n];
        }
        S.blk[i].fc2cat = P.linear_raw(wc.data(), bc.data(), C, hid + Cp);
      }
    }
    S.norm = P.norm("norm" + sn, C);
  }
  // flow encoder: conv + BN(eval) folded, ReLU applied in the GEMM epilogue
  const int fch[5] = {2, 64, 128, c.embed_dims[2], c.embed_dims[3]};
  for (int i = 0; i < 4; ++i) {
    std::vector<float> sc, sh;
    const std::string n = std::to_string(i + 1);
    if (P.bn("flow_encoder.bn" + n, fch[i + 1], &sc, &sh)) h->flow[i] = P.conv("flow_encoder.conv" + n, fch[i + 1], fch[i], i == 0 ? 7 : 3, sc.data(), sh.data());
  }
  // cross attention: in_proj_weight rows = [Wq; Wk; Wv]
  for (int j = 0; j < 2; ++j) {
    const int C = c.embed_dims[2 + j];
    const std::string p = "cross_attn_s" + std::to_string(3 + j);
    const HostTensor* w = P.get(p + ".cross_attn.in_proj_weight", {3 * C, C});
    const HostTensor* b = P.get(p + ".cross_attn.in_proj_bias", {3 * C});
    if (w && b) {
      h->xa[j].q = P.linear_raw(w->data.data(), b->data.data(), C, C);
      h->xa[j].kv = P.linear_raw(w->data.data() + static_cast<size_t>(C) * C, b->data.data() + C, 2 * C, C);
    }
    h->xa[j].out = P.linear(p + ".cross_attn.out_proj", C, C);
    h->xa[j].norm = P.norm(p + ".norm", C);
  }
  // head
  std::vector<float> sc, sh;
  const bool have_bn = P.bn("head.linear_fuse.bn", E, &sc, &sh);
  const HostTensor* wf = P.get("head.linear_fuse.conv.weight", {E, 4 * E, 1, 1});
  for (int i = 0; i < 4; ++i) h->head_c[i] = P.linear("head.linear_c" + std::to_string(i + 1) + ".proj", E, c.embed_dims[i]);
  if (have_bn && wf) {
    h->head_fuse = P.linear_raw(wf->data.data(), sh.data(), E, 4 * E, sc.data());
    if (c.fold_head && P.err.empty()) {
      // W'[:, blk_i] = diag(scale) W_fuse[:, blk_i] W_c_i ; b' = diag(scale) sum_i W_fuse[:, blk_i] b_c_i + shift.
      // concat order along K is [c4, c3, c2, c1] (segformer_head.py:158).
      int Ktot = 0;
      for (int i = 0; i < 4; ++i) Ktot += c.embed_dims[i];
      std::vector<float> Wp(static_cast<size_t>(E) * Ktot), bp(E);
      std::vector<double> acc;
      int koff = 0;
      std::vector<double> bacc(E, 0.0);
      for (int blk = 0; blk < 4; ++blk) {
        const int ci = 3 - blk;  // c4 first
        const int Ci = c.embed_dims[ci];
        const HostTensor* wc = P.get("head.linear_c" + std::to_string(ci + 1) + ".proj.weight", {E, Ci});
        const HostTensor* bc = P.get("head.linear_c" + std::to_string(ci + 1) + ".proj.bias", {E});
        if (!wc || !bc) break;
        for (int o = 0; o < E; ++o) {
          acc.assign(Ci, 0.0);
          const float* wrow = wf->data.data() + static_cast<size_t>(o) * 4 * E + static_cast<size_t>(blk) * E;
          double bsum = 0.0;
          for (int e = 0; e < E; ++e) {
            const double wv = wrow[e];
            const float* wcr = wc->data.data() + static_cast<size_t>(e) * Ci;
            for (int k = 0; k < Ci; ++k) acc[k] += wv * wcr[k];
            bsum += wv * bc->data[e];
          }
          for (int k = 0; k < Ci; ++k) Wp[static_cast<size_t>(o) * Ktot + koff + k] = static_cast<float>(acc[k]);
          bacc[o] += bsum;
        }
        koff += Ci;
      }
      for (int o = 0; o < E; ++o) bp[o] = static_cast<float>(bacc[o] * sc[o] + sh[o]);
      h->head_fold = P.linear_raw(Wp.data(), bp.data(), E, Ktot, sc.data());
    }
  }
  // fp32 classifier heads (segformer_head.py:101-106)
  const char* fcn[2] = {"head.fc", "head.fc_ant"};
  for (int a = 0; a < 2; ++a) {
    const HostTensor* w0 = P.get(std::string(fcn[a]) + ".0.weight", {512, 2048});
    const HostTensor* w2 = P.get(std::string(fcn[a]) + ".2.weight", {7, 512});
    h->fc_w[a][0] = P.alloc_f(512 * 2048);
    h->fc_w[a][1] = P.alloc_f(7 * 512);
    if (w0) std::copy(w0->data.begin(), w0->data.end(), P.wf.begin() + h->fc_w[a][0]);
    if (w2) std::copy(w2->data.begin(), w2->data.end(), P.wf.begin() + h->fc_w[a][1]);
    h->fc_b[a][0] = P.vec(std::string(fcn[a]) + ".0.bias", 512);
    h->fc_b[a][1] = P.vec(std::string(fcn[a]) + ".2.bias", 7);
  }
  if (!P.err.empty()) return fail(SV_ERR_STATE, P.err);

  SV_TRY(upload(h->device, &h->d_wb, P.wb));
  SV_TRY(upload(h->device, &h->d_wf, P.wf));
  h->plans.clear();
  h->last_plan = nullptr;
  h->sd.packed = true;
  return SV_OK;
}

// --------------------------------------------------------------------------------------------- geometry
void stage_geometry(const sv_evp_cfg& c, int H, int W, StageGeom (&g)[4]) {
  const int ks[4] = {7, 3, 3, 3}, st[4] = {4, 2, 2, 2};
  int h = H, w = W;
  for (int s = 0; s < 4; ++s) {
    h = conv_out_dim(h, ks[s], st[s], ks[s] / 2);
    w = conv_out_dim(w, ks[s], st[s], ks[s] / 2);
    StageGeom& G = g[s];
    G.H = h; G.W = w; G.N = h * w; G.C = c.embed_dims[s]; G.heads = c.num_heads[s]; G.sr = c.sr_ratios[s];
    G.Hk = G.sr > 1 ? conv_out_dim(h, G.sr, G.sr, 0) : h;
    G.Wk = G.sr > 1 ? conv_out_dim(w, G.sr, G.sr, 0) : w;
    G.Nkv = G.Hk * G.Wk;
    G.hidden = G.C * c.mlp_ratio;
    G.Cp = G.C / 4;
  }
}

// stage_geometry of a checked config and input size (the host-only queries take the config from the caller)
int pyramid(const sv_evp_cfg& c, int H, int W, StageGeom (&g)[4]) {
  if (H <= 0 || W <= 0) return fail(SV_ERR_INVALID, "evp: H and W must be positive");
  for (int s = 0; s < 4; ++s)
    if (c.embed_dims[s] <= 0 || c.num_heads[s] <= 0 || c.depths[s] <= 0 || c.sr_ratios[s] <= 0 || c.embed_dims[s] % c.num_heads[s] != 0)
      return fail(SV_ERR_INVALID, "evp: bad config (non-positive entry or dim not divisible by heads)");
  stage_geometry(c, H, W, g);
  for (int s = 0; s < 4; ++s)
    if (g[s].H < 1 || g[s].W < 1 || g[s].Hk < 1 || g[s].Wk < 1) return fail(SV_ERR_INVALID, "evp: input too small for the 4-stage pyramid");
  return SV_OK;
}

// pyramid() for forward_features, which also rejects what the reference's forward_features cannot run: a stage map smaller than
// its spatial-reduction window (Conv2d(kernel = stride = sr) raises there; at 224 / 4 / 8 / ... the smallest input is 29 x 29)
int features_pyramid(const sv_evp_cfg& c, int H, int W, StageGeom (&g)[4]) {
  SV_TRY(pyramid(c, H, W, g));
  for (int s = 0; s < 4; ++s)
    if (g[s].sr > 1 && (g[s].H < g[s].sr || g[s].W < g[s].sr))
      return fail(SV_ERR_INVALID, "evp: input too small for the 4-stage pyramid: stage " + std::to_string(s + 1) + " is " + std::to_string(g[s].H) +
                                      "x" + std::to_string(g[s].W) + ", smaller than its spatial-reduction window " + std::to_string(g[s].sr));
  return SV_OK;
}

// Where each encoder block's attention maps [B, heads, N, N_kv] (fp32) go in one buffer, in call order (stage 1 blocks first).
// off has n_blocks + 1 entries (element offsets; the last is the total), dims 3 per block.
int maps_layout(const sv_evp_cfg& c, int B, int H, int W, std::vector<int64_t>* off, std::vector<int32_t>* dims) {
  if (B <= 0 || H <= 0 || W <= 0) return fail(SV_ERR_INVALID, "evp: B, H and W must be positive");
  StageGeom g[4];
  SV_TRY(pyramid(c, H, W, g));
  off->assign(1, 0);
  dims->clear();
  for (int s = 0; s < 4; ++s)
    for (int i = 0; i < c.depths[s]; ++i) {
      off->push_back(off->back() + static_cast<int64_t>(B) * g[s].heads * g[s].N * g[s].Nkv);
      dims->insert(dims->end(), {g[s].heads, g[s].N, g[s].Nkv});
    }
  return SV_OK;
}

// --------------------------------------------------------------------------------------------- plan building
struct Builder {
  sv_evp* h;
  Plan* plan;      // nullptr in dry (sizing) mode
  Arena arena;
  int status = SV_OK;
  Builder(sv_evp* hh, Plan* p, void* ws) : h(hh), plan(p), arena(ws) {}
  bool dry() const { return plan == nullptr; }
  const bf16* W(const Lin& l) const { return h->d_wb + l.w; }
  const float* Bf(const Lin& l) const { return l.has_bias ? h->d_wf + l.b : nullptr; }
  const float* F(size_t off) const { return h->d_wf + off; }

  template <typename R>
  void push(const R& rec, double alg_bytes) {
    if (dry() || status != SV_OK) return;
    plan->ops.push_back(Op{rec, alg_bytes});
    plan->bytes_by_kind[R::kind] += alg_bytes;
  }
  // the step gemm() and conv() share: the result and the A operand (a_bytes from d.A) must lie inside one workspace buffer each
  void push_gemm(const GemmDesc& d, size_t a_bytes, double alg_bytes, const char* bounds_error) {
    if (dry() || status != SV_OK) return;
    if (!arena.contains(d.out, (static_cast<size_t>(d.M - 1) * d.ldc + d.N) * (d.out_fp32 ? 4 : 2)) || !arena.contains(d.A, a_bytes)) {
      status = fail(SV_ERR_STATE, bounds_error);
      return;
    }
    GemmOp op;
    status = gemm_plan(d, &op.plan);
    plan->gemm_flops += op.plan.flops;
    push(op, alg_bytes);
  }

  // A2/lda2/K2: optional second A segment for the last K2 columns of K (see GemmDesc)
  void gemm(const bf16* A, int64_t lda, const Lin& l, int M, int act, const float* resid, int64_t ldr, void* out, int64_t ldc, int out_fp32,
            const bf16* A2 = nullptr, int64_t lda2 = 0, int K2 = 0) {
    GemmDesc d;
    d.A = A; d.lda = lda; d.W = W(l); d.ldw = l.ldw; d.M = M; d.N = l.N; d.bias = Bf(l); d.act = act;
    d.A2 = A2; d.lda2 = lda2; d.K2 = K2;
    d.K = l.ldw;  // K padded to a multiple of 8; pad columns are zero in both the packed weight and the im2col buffer
    d.residual = resid; d.ldr = ldr; d.out = out; d.ldc = ldc; d.out_fp32 = out_fp32;
    push_gemm(d, (static_cast<size_t>(M - 1) * lda + (l.ldw - K2)) * 2,
              2.0 * M * d.K + 2.0 * l.N * d.K + static_cast<double>(M) * l.N * (out_fp32 ? 4 : 2) + (resid ? 4.0 * M * l.N : 0.0),
              "evp: internal error: a GEMM of the plan addresses memory outside its workspace buffer");
  }
  // convolution of an NHWC bf16 input with (kh, kw, cin)-packed weights: an implicit GEMM whose A tiles the TMA gathers through an
  // im2col-mode map when the geometry allows (conv_gemm_im2col_ok), else an im2col gather into `col` and a GEMM over it
  void conv(const bf16* x, const ConvGeom& cg, const Lin& l, int act, void* out, int64_t ldc, int out_fp32, bf16* col) {
    const int M = cg.B * cg.Ho() * cg.Wo();
    if (!conv_gemm_im2col_ok(cg)) {
      im2col(EXT_NONE, nullptr, x, cg.B, cg.C, cg.H, cg.W, cg.k, cg.stride, cg.pad, col, l.ldw);
      gemm(col, l.ldw, l, M, act, nullptr, 0, out, ldc, out_fp32);
      return;
    }
    const size_t x_bytes = static_cast<size_t>(cg.B) * cg.H * cg.W * cg.C * 2;
    GemmDesc d;
    d.A = x; d.conv = cg; d.W = W(l); d.ldw = l.ldw; d.M = M; d.N = l.N; d.K = l.ldw; d.bias = Bf(l); d.act = act;
    d.out = out; d.ldc = ldc; d.out_fp32 = out_fp32;
    push_gemm(d, x_bytes, static_cast<double>(x_bytes) + 2.0 * l.N * d.K + static_cast<double>(M) * l.N * (out_fp32 ? 4 : 2),
              "evp: internal error: a conv GEMM of the plan addresses memory outside its workspace buffer");
  }
  void ln(const float* x, const Norm& n, float eps, int64_t rows, float* of, bf16* ob, bf16* patch = nullptr, int pH = 0, int pW = 0, int psr = 0) {
    push(LayerNormOp{x, F(n.g), F(n.b), eps, rows, n.C, of, ob, patch, pH, pW, psr},
         static_cast<double>(rows) * n.C * (4 + (of ? 4 : 0) + (ob ? 2 : 0) + (patch ? 2 : 0)));
  }
  void im2col(Ext ext, const float* nchw, const bf16* nhwc, int B, int Cin, int H, int W, int k, int stride, int pad, bf16* out, int64_t ldo) {
    push(Im2colOp{ext, nchw, nhwc, B, Cin, H, W, k, stride, pad, out, ldo},
         static_cast<double>(B) * Cin * H * W * (nhwc ? 2 : 4) +
             2.0 * B * conv_out_dim(H, k, stride, pad) * conv_out_dim(W, k, stride, pad) * static_cast<double>(ldo));
  }
  void dwconv(const bf16* x, size_t w, size_t b, int B, int H, int W, int C, bf16* out, int64_t ldo) {
    if (dry() || status != SV_OK) return;
    const double bytes = 2.0 * 2.0 * B * H * W * static_cast<double>(C);
    if (!dwconv_tma_supported(C)) return push(DwconvOp{x, F(w), F(b), B, H, W, C, out, ldo}, bytes);
    DwconvTmaOp op;
    status = dwconv_tma_plan(x, F(w), F(b), B, H, W, C, out, ldo, &op.plan);
    push(op, bytes);
  }
  void attn(const bf16* q, int64_t ldq, const bf16* k, int64_t ldk, const bf16* v, int64_t ldv, bf16* o, int64_t ldo, int B, int heads, int Nq, int Nkv, int hd) {
    if (dry() || status != SV_OK) return;
    const float scale = 1.0f / sqrtf(static_cast<float>(hd));
    const double bytes = 2.0 * B * heads * hd * (2.0 * Nq + 2.0 * Nkv);
    if (!attention_tc_enabled() || !attention_tc_supported(hd, Nkv, ldq, ldk, ldv, ldo, q, k, v, o))
      return push(AttnOp{q, ldq, k, ldk, v, ldv, o, ldo, B, heads, Nq, Nkv, hd, scale}, bytes);
    AttnTcOp op{{}, ldq, hd};
    status = attention_tc_plan(q, ldq, k, ldk, v, ldv, o, ldo, B, heads, Nq, Nkv, scale, &op.plan);
    push(op, bytes);
  }
  // P = softmax(Q K^T * scale) of encoder block `block` into the caller's maps buffer (resolved per call, see run_plan)
  void probs(const bf16* q, int64_t ldq, const bf16* k, int64_t ldk, int B, int heads, int Nq, int Nkv, int hd, int block) {
    push(ProbsOp{q, ldq, k, ldk, B, heads, Nq, Nkv, hd, 1.0f / sqrtf(static_cast<float>(hd)), block},
         2.0 * B * heads * hd * (static_cast<double>(Nq) + Nkv) + 4.0 * B * heads * static_cast<double>(Nq) * Nkv);
  }
  // stage norm of the encoder-only plans: channel-major fp32 into the caller's stage_out[stage] (resolved per call, see run_plan)
  void stage_norm(const float* x, const Norm& n, float eps, int64_t rows, int tokens, bf16* ob, int stage) {
    push(StageNormOp{x, F(n.g), F(n.b), eps, rows, n.C, tokens, ob, stage}, static_cast<double>(rows) * n.C * (4 + 4 + 2));
  }
  void gauss(float* out, int planes, int H, int W) { push(GaussOp{out, planes, H, W}, 8.0 * planes * H * W); }
  void bilinear(const bf16* x, int B, int H, int W, int C, int Ho, int Wo, bf16* out, int64_t ldo) { push(BilinearOp{x, B, H, W, C, Ho, Wo, out, ldo}, 0.0); }
  void mean(const float* x, int B, int tokens, int C) { push(MeanOp{x, B, tokens, C}, 0.0); }
  // fused k7s4p3 conv on an fp32 NCHW input + LayerNorm (norm != nullptr) or ReLU
  void stem(Ext ext, const float* src, const Lin& l, const Norm* norm, int B, int Cin, int H, int W, float* of, bf16* ob) {
    const double outpx = static_cast<double>(B) * conv_out_dim(H, 7, 4, 3) * conv_out_dim(W, 7, 4, 3);
    push(StemOp{ext, src, this->W(l), l.ldw, Bf(l), norm ? F(norm->g) : nullptr, norm ? F(norm->b) : nullptr, 1e-5f, norm ? 0 : 1, B, Cin, H, W, l.N, of, ob},
         4.0 * B * Cin * H * W + outpx * l.N * ((of ? 4 : 0) + (ob ? 2 : 0)));
  }
  void tap(const std::string& name, const bf16* p, int64_t elems) { if (!dry()) plan->taps[name] = Tap{p, elems}; }
};

// MotionGuidedCrossAttention is nn.MultiheadAttention(dim, 8 heads) (mix_transformer_evp.py:866-870): C/8 of stages 3 and 4 is its head_dim
bool flow_supported(const sv_evp_cfg& c) {
  for (int j = 2; j < 4; ++j) {
    const int hd = c.embed_dims[j] / 8;
    if (c.embed_dims[j] % 8 != 0 || (hd != 20 && hd != 32 && hd != 40 && hd != 64)) return false;
  }
  return true;
}

// Builds (or only sizes, when plan == nullptr) the launch schedule for n frames of HxW.  features_only: the encoder-only plan of
// forward_features, which ends with the stage norms writing the call's fp32 NCHW stage maps (no flow branch, no head); it addresses a
// prefix of the workspace of the full plan without flow.
int build(sv_evp* h, Plan* plan, void* ws, int n, int H, int W, bool with_flow, bool capture, bool features_only, size_t* bytes_out) {
  const sv_evp_cfg& c = h->cfg;
  Builder b(h, plan, ws);
  Arena& A = b.arena;
  StageGeom g[4];
  stage_geometry(c, H, W, g);
  for (int s = 0; s < 4; ++s) {
    if (g[s].H < 1 || g[s].W < 1 || g[s].Hk < 1 || g[s].Wk < 1) return fail(SV_ERR_INVALID, "evp: input too small for the 4-stage pyramid");
  }
  if (with_flow && !flow_supported(c)) return fail(SV_ERR_UNSUPPORTED, "evp: flow cross-attention head_dim (C/8) must be 20, 32, 40 or 64");
  const int E = c.embedding_dim;
  const int ks[4] = {7, 3, 3, 3}, strd[4] = {4, 2, 2, 2};
  const int fch[5] = {2, 64, 128, c.embed_dims[2], c.embed_dims[3]};
  auto geom = [&](int B, int Hi, int Wi, int C, int k, int st, int pad) {
    ConvGeom cg;
    cg.B = B; cg.H = Hi; cg.W = Wi; cg.C = C; cg.k = k; cg.stride = st; cg.pad = pad;
    return cg;
  };
  // does the stage-s conv (patch embed / handcrafted prompt / flow conv, input width cin) gather an im2col buffer?  Stage 0 runs the
  // fused stem when it can (the same test as below, on the packed shapes), stages 1-3 read their input through an im2col map when they can
  auto needs_col = [&](int s, int cin, int cout) {
    if (s == 0) return !stem_conv_supported(cin, cout, round_up(49 * cin, 8));
    return !conv_gemm_im2col_ok(geom(n, g[s - 1].H, g[s - 1].W, cin, 3, 2, 1));
  };

  // ---- sizes of stage-scoped buffers (max over stages)
  size_t max_tok_c = 0, max_tok_cp = 0, max_tok_hid = 0, max_tok_tall = 0, max_kv_c = 0, max_sr_k = 0, max_col = 0, max_conv_out = 0;
  for (int s = 0; s < 4; ++s) {
    const size_t M = static_cast<size_t>(n) * g[s].N, Mk = static_cast<size_t>(n) * g[s].Nkv;
    max_tok_c = std::max(max_tok_c, M * g[s].C);
    max_tok_cp = std::max(max_tok_cp, M * g[s].Cp);
    max_tok_hid = std::max(max_tok_hid, M * g[s].hidden);
    max_tok_tall = std::max(max_tok_tall, M * static_cast<size_t>(c.depths[s]) * g[s].Cp);
    max_kv_c = std::max(max_kv_c, Mk * g[s].C);
    if (g[s].sr > 1 && !conv_gemm_im2col_ok(geom(n, g[s].H, g[s].W, g[s].C, g[s].sr, g[s].sr, 0)))   // LN1's sr-patch copy
      max_sr_k = std::max(max_sr_k, Mk * static_cast<size_t>(g[s].sr * g[s].sr * g[s].C));
    const int cin = s == 0 ? 3 : c.embed_dims[s - 1];
    const int cinp = s == 0 ? 3 : c.embed_dims[s - 1] / 4;
    if (needs_col(s, cin, g[s].C)) max_col = std::max(max_col, M * static_cast<size_t>(round_up(ks[s] * ks[s] * cin, 8)));
    if (needs_col(s, cinp, g[s].Cp)) max_col = std::max(max_col, M * static_cast<size_t>(round_up(ks[s] * ks[s] * cinp, 8)));
    max_conv_out = std::max(max_conv_out, M * g[s].C);
  }
  // the flow cross-attention keys/values cover the stage's FULL token grid (no spatial reduction): [n*N, 2C] in `kvb`
  if (with_flow)
    for (int s = 2; s < 4; ++s) max_kv_c = std::max(max_kv_c, static_cast<size_t>(n) * g[s].N * g[s].C);
  if (with_flow)
    for (int i = 0; i < 4; ++i)
      if (needs_col(i, fch[i], fch[i + 1])) max_col = std::max(max_col, static_cast<size_t>(n) * g[i].N * round_up((i == 0 ? 49 : 9) * fch[i], 8));

  // ---- buffers
  float* seg_g = A.get<float>(static_cast<size_t>(n) * 3 * H * W);
  bf16* col = max_col > 0 ? A.get<bf16>(max_col) : nullptr;
  float* conv_out = A.get<float>(max_conv_out);
  float* hc_f32[4];
  bf16* hc_b16[4];
  bf16* c_b16[4];
  float* c_f32[4] = {nullptr, nullptr, nullptr, nullptr};
  for (int s = 0; s < 4; ++s) {
    const size_t M = static_cast<size_t>(n) * g[s].N;
    hc_f32[s] = A.get<float>(M * g[s].Cp);
    hc_b16[s] = A.get<bf16>(M * g[s].Cp);
    c_b16[s] = A.get<bf16>(M * g[s].C);
    if (s >= 2 && with_flow) c_f32[s] = A.get<float>(M * g[s].C);
  }
  float* x = A.get<float>(max_tok_c);
  bf16* xn = A.get<bf16>(max_tok_c);
  bf16* qb = A.get<bf16>(max_tok_c);
  bf16* ob = A.get<bf16>(max_tok_c);
  bf16* Pb = A.get<bf16>(max_tok_cp);
  bf16* a_sr = max_sr_k > 0 ? A.get<bf16>(max_sr_k) : nullptr;   // sr-patch copy of LN1, only for sr convs without an im2col map
  float* sr_out = A.get<float>(max_kv_c);
  bf16* srn = A.get<bf16>(max_kv_c);
  bf16* kvb = A.get<bf16>(2 * max_kv_c);
  bf16* h1 = A.get<bf16>(max_tok_hid);
  bf16* h2 = A.get<bf16>(max_tok_hid);     // [M, 4C]: GELU(dwconv(h1))
  bf16* T_all = A.get<bf16>(max_tok_tall);  // [M, depth * C/4]: GELU(lightweight_mlp_i(P)) for every block i of the stage

  // ---- 0. handcrafted prompts: gaussian(seg) -> 4 chained OverlapPatchEmbeds (mix_transformer_evp.py:718-747)
  b.gauss(seg_g, n * 3, H, W);
  {
    int hh = H, ww = W;
    for (int s = 0; s < 4; ++s) {
      const int cinp = s == 0 ? 3 : c.embed_dims[s - 1] / 4;
      const StageW& S = h->st[s];
      const int M = n * g[s].N;
      if (s == 0 && stem_conv_supported(cinp, S.hc.N, S.hc.ldw)) {
        b.stem(EXT_NONE, seg_g, S.hc, &S.hc_norm, n, cinp, hh, ww, hc_f32[s], hc_b16[s]);
      } else {
        if (s == 0) {
          b.im2col(EXT_NONE, seg_g, nullptr, n, cinp, hh, ww, ks[s], strd[s], ks[s] / 2, col, S.hc.ldw);
          b.gemm(col, S.hc.ldw, S.hc, M, ACT_NONE, nullptr, 0, conv_out, g[s].Cp, 1);
        } else {
          b.conv(hc_b16[s - 1], geom(n, hh, ww, cinp, ks[s], strd[s], ks[s] / 2), S.hc, ACT_NONE, conv_out, g[s].Cp, 1, col);
        }
        b.ln(conv_out, S.hc_norm, 1e-5f, M, hc_f32[s], hc_b16[s]);
      }
      hh = g[s].H; ww = g[s].W;
    }
  }
  // ---- 1. encoder stages
  {
    int hh = H, ww = W;
    int block = 0;  // encoder block index over all stages (capture plans)
    for (int s = 0; s < 4; ++s) {
      const StageGeom& G = g[s];
      const StageW& S = h->st[s];
      const int M = n * G.N, Mk = n * G.Nkv, C = G.C;
      const int cin = s == 0 ? 3 : c.embed_dims[s - 1];
      if (s == 0 && stem_conv_supported(cin, S.pe.N, S.pe.ldw)) {
        b.stem(EXT_X, nullptr, S.pe, &S.pe_norm, n, cin, hh, ww, x, xn);
      } else {
        if (s == 0) {
          b.im2col(EXT_X, nullptr, nullptr, n, cin, hh, ww, ks[s], strd[s], ks[s] / 2, col, S.pe.ldw);
          b.gemm(col, S.pe.ldw, S.pe, M, ACT_NONE, nullptr, 0, conv_out, C, 1);
        } else {
          b.conv(c_b16[s - 1], geom(n, hh, ww, cin, ks[s], strd[s], ks[s] / 2), S.pe, ACT_NONE, conv_out, C, 1, col);
        }
        b.ln(conv_out, S.pe_norm, 1e-5f, M, x, xn);
      }
      // init_prompt (:749-756): P = handcrafted_s + embedding_generator_s(x)   (constant over depth)
      b.gemm(xn, C, S.emb, M, ACT_NONE, hc_f32[s], G.Cp, Pb, G.Cp, 0);
      const int ldh = G.hidden;
      const int ldt = c.depths[s] * G.Cp;
      // every block's T_i = GELU(lightweight_mlp_i(P)) in one GEMM (P is constant over the depth of the stage)
      b.gemm(Pb, G.Cp, S.lw_all, M, ACT_GELU, nullptr, 0, T_all, ldt, 0);
      for (int i = 0; i < c.depths[s]; ++i) {
        const BlockW& Bk = S.blk[i];
        const bool has_next = i + 1 < c.depths[s];
        // get_prompt (:776-815): x += shared_mlp(T_i).  Only block 0 does this as its own GEMM; for i >= 1 the term was already
        // added by block i-1's K-concatenated fc2 GEMM (see pack_all).
        if (i == 0) b.gemm(T_all, ldt, S.shared, M, ACT_NONE, x, C, x, C, 1);
        // attention (:110-131).  The sr conv (k = stride = sr, no padding) reads LN1's output through an im2col map; where it cannot,
        // LN1 also emits the conv's A operand (non-overlapping sr x sr patches) as a second bf16 copy
        if (G.sr > 1) {
          const ConvGeom srg = geom(n, G.H, G.W, C, G.sr, G.sr, 0);
          const bool sr_map = conv_gemm_im2col_ok(srg);
          b.ln(x, Bk.n1, 1e-6f, M, nullptr, xn, sr_map ? nullptr : a_sr, G.H, G.W, G.sr);
          b.gemm(xn, C, Bk.q, M, ACT_NONE, nullptr, 0, qb, C, 0);
          if (sr_map) b.conv(xn, srg, Bk.sr, ACT_NONE, sr_out, C, 1, nullptr);
          else b.gemm(a_sr, Bk.sr.ldw, Bk.sr, Mk, ACT_NONE, nullptr, 0, sr_out, C, 1);
          b.ln(sr_out, Bk.srn, 1e-5f, Mk, nullptr, srn);
          b.gemm(srn, C, Bk.kv, Mk, ACT_NONE, nullptr, 0, kvb, 2 * C, 0);
        } else {
          b.ln(x, Bk.n1, 1e-6f, M, nullptr, xn);
          b.gemm(xn, C, Bk.q, M, ACT_NONE, nullptr, 0, qb, C, 0);
          b.gemm(xn, C, Bk.kv, M, ACT_NONE, nullptr, 0, kvb, 2 * C, 0);
        }
        b.attn(qb, C, kvb, 2 * C, kvb + C, 2 * C, ob, C, n, G.heads, G.N, G.Nkv, C / G.heads);
        if (capture) b.probs(qb, C, kvb, 2 * C, n, G.heads, G.N, G.Nkv, C / G.heads, block);
        ++block;
        b.gemm(ob, C, Bk.proj, M, ACT_NONE, x, C, x, C, 1);
        // MixFFN (:60-67)
        b.ln(x, Bk.n2, 1e-6f, M, nullptr, xn);
        b.gemm(xn, C, Bk.fc1, M, ACT_NONE, nullptr, 0, h1, G.hidden, 0);
        b.dwconv(h1, Bk.dw_w, Bk.dw_b, n, G.H, G.W, G.hidden, h2, ldh);
        if (has_next) {
          // x += fc2(h) + shared_mlp(T_{i+1}): A = [h2 | T_{i+1}] as two K segments, W = [W_fc2 | W_shared]
          b.gemm(h2, ldh, Bk.fc2cat, M, ACT_NONE, x, C, x, C, 1, T_all + static_cast<size_t>(i + 1) * G.Cp, ldt, G.Cp);
        } else {
          b.gemm(h2, ldh, Bk.fc2, M, ACT_NONE, x, C, x, C, 1);
        }
      }
      if (features_only) b.stage_norm(x, S.norm, 1e-6f, M, G.N, c_b16[s], s);
      else b.ln(x, S.norm, 1e-6f, M, c_f32[s], c_b16[s]);
      b.tap("stage" + std::to_string(s + 1) + "_tokens", c_b16[s], static_cast<int64_t>(M) * C);
      hh = G.H; ww = G.W;
    }
  }
  if (features_only) {
    if (bytes_out) *bytes_out = ((A.off + 255) & ~static_cast<size_t>(255)) + 256;
    return b.status;
  }
  // ---- 2. optical-flow branch (:423-444)
  const bf16* head_in[4] = {c_b16[0], c_b16[1], c_b16[2], c_b16[3]};
  if (with_flow) {
    bf16* fl[4];
    for (int i = 0; i < 4; ++i) fl[i] = A.get<bf16>(static_cast<size_t>(n) * g[i].N * fch[i + 1]);
    int hh = H, ww = W;
    for (int i = 0; i < 4; ++i) {
      const Lin& L = h->flow[i];
      const int M = n * g[i].N;
      if (i == 0 && stem_conv_supported(2, L.N, L.ldw)) {
        b.stem(EXT_FLOW, nullptr, L, nullptr, n, 2, hh, ww, nullptr, fl[i]);
      } else {
        if (i == 0) {
          b.im2col(EXT_FLOW, nullptr, nullptr, n, 2, hh, ww, 7, 4, 3, col, L.ldw);
          b.gemm(col, L.ldw, L, M, ACT_RELU, nullptr, 0, fl[i], fch[i + 1], 0);
        } else {
          b.conv(fl[i - 1], geom(n, hh, ww, fch[i], 3, 2, 1), L, ACT_RELU, fl[i], fch[i + 1], 0, col);
        }
      }
      hh = g[i].H; ww = g[i].W;
    }
    for (int j = 0; j < 2; ++j) {
      const int s = 2 + j;
      const StageGeom& G = g[s];
      const CrossW& X = h->xa[j];
      const int M = n * G.N, C = G.C;
      bf16* fused = A.get<bf16>(static_cast<size_t>(M) * C);
      b.gemm(c_b16[s], C, X.q, M, ACT_NONE, nullptr, 0, qb, C, 0);
      b.gemm(fl[s], C, X.kv, M, ACT_NONE, nullptr, 0, kvb, 2 * C, 0);   // flow tokens share the stage's grid
      b.attn(qb, C, kvb, 2 * C, kvb + C, 2 * C, ob, C, n, 8, G.N, G.N, C / 8);
      b.gemm(ob, C, X.out, M, ACT_NONE, c_f32[s], C, x, C, 1);          // x_visual + out_proj(attn)
      b.ln(x, X.norm, 1e-5f, M, nullptr, fused);
      b.tap("fused" + std::to_string(s + 1) + "_tokens", fused, static_cast<int64_t>(M) * C);
      head_in[s] = fused;
    }
  }
  // ---- 3. SegFormer head (segformer_head.py:137-173).  The per-pixel affine linear_c{i} commutes with the bilinear
  // resize (its weights sum to 1), so c1..c3 are resized to c4's grid FIRST and projected on 49 tokens/frame.
  {
    const int Ho = g[3].H, Wo = g[3].W, M4 = n * Ho * Wo;
    int Ktot = 0;
    for (int i = 0; i < 4; ++i) Ktot += c.embed_dims[i];
    float* y = A.get<float>(static_cast<size_t>(M4) * E);
    if (c.fold_head) {
      bf16* pooled = A.get<bf16>(static_cast<size_t>(M4) * Ktot);
      int koff = 0;
      for (int blk = 0; blk < 4; ++blk) {
        const int ci = 3 - blk;
        b.bilinear(head_in[ci], n, g[ci].H, g[ci].W, g[ci].C, Ho, Wo, pooled + koff, Ktot);
        koff += g[ci].C;
      }
      b.gemm(pooled, Ktot, h->head_fold, M4, ACT_RELU, nullptr, 0, y, E, 1);
    } else {
      bf16* cat = A.get<bf16>(static_cast<size_t>(M4) * 4 * E);
      bf16* pooled = A.get<bf16>(static_cast<size_t>(M4) * c.embed_dims[3]);
      for (int blk = 0; blk < 4; ++blk) {
        const int ci = 3 - blk;
        const bf16* src = head_in[ci];
        if (ci != 3) {
          b.bilinear(head_in[ci], n, g[ci].H, g[ci].W, g[ci].C, Ho, Wo, pooled, g[ci].C);
          src = pooled;
        }
        b.gemm(src, g[ci].C, h->head_c[ci], M4, ACT_NONE, nullptr, 0, cat + static_cast<size_t>(blk) * E, 4 * E, 0);
      }
      b.gemm(cat, 4 * E, h->head_fuse, M4, ACT_RELU, nullptr, 0, y, E, 1);  // conv1x1 (BN folded) + ReLU
    }
    b.mean(y, n, Ho * Wo, E);  // Dropout2d = identity in eval; AdaptiveAvgPool2d(1); flatten
  }
  if (bytes_out) *bytes_out = ((A.off + 255) & ~static_cast<size_t>(255)) + 256;
  return b.status;
}

int run_plan(sv_evp* h, const Plan& p, const CallIO& io, cudaStream_t st) {
  const bool prof = h->profile;
  if (prof) {
    while (h->prof_events.size() < 2 * p.ops.size()) {
      cudaEvent_t e;
      SV_CUDA_OK(cudaEventCreate(&e));
      h->prof_events.push_back(e);
    }
  }
  size_t op_idx = 0;
  for (const Op& op : p.ops) {
    if (prof) SV_CUDA_OK(cudaEventRecord(h->prof_events[2 * op_idx], st));
    const int rc = std::visit([&](const auto& r) { return r.launch(io, st); }, op.rec);
    if (rc != SV_OK) return rc;
    if (prof) SV_CUDA_OK(cudaEventRecord(h->prof_events[2 * op_idx + 1], st));
    ++op_idx;
    ++h->launches;
  }
  if (prof) {
    SV_CUDA_OK(cudaStreamSynchronize(st));
    for (size_t i = 0; i < p.ops.size(); ++i) {
      float ms = 0.f;
      SV_CUDA_OK(cudaEventElapsedTime(&ms, h->prof_events[2 * i], h->prof_events[2 * i + 1]));
      h->prof_ms[p.ops[i].kind()] += ms;
      h->prof_n[p.ops[i].kind()] += 1;
      p.ops[i].prof_ms += ms;
      p.ops[i].prof_n += 1;
    }
    h->prof_gemm_flops += p.gemm_flops;
    for (int i = 0; i < OP_KINDS; ++i) h->prof_bytes[i] += p.bytes_by_kind[i];
  }
  return SV_OK;
}

// fp32 classifier MLP: one block per frame; warp-per-output dot products
__global__ void __launch_bounds__(512) classify_kernel(const float* __restrict__ feats, const float* __restrict__ w0, const float* __restrict__ b0,
                                                       const float* __restrict__ w2, const float* __restrict__ b2, float* __restrict__ out) {
  __shared__ float hid[512];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float* f = feats + static_cast<int64_t>(blockIdx.x) * 2048;
  for (int o = warp; o < 512; o += 16) {
    const float* w = w0 + static_cast<int64_t>(o) * 2048;
    float s = 0.f;
    for (int k = lane * 4; k < 2048; k += 128) {
      const float4 a = *reinterpret_cast<const float4*>(f + k);
      const float4 b = __ldg(reinterpret_cast<const float4*>(w + k));
      s += a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w;
    }
    s = warp_sum(s);
    if (lane == 0) hid[o] = fmaxf(s + b0[o], 0.f);
  }
  __syncthreads();
  if (warp < 7) {
    float s = 0.f;
    for (int k = lane; k < 512; k += 32) s += hid[k] * w2[warp * 512 + k];
    s = warp_sum(s);
    if (lane == 0) out[static_cast<int64_t>(blockIdx.x) * 7 + warp] = s + b2[warp];
  }
}

}  // namespace
}  // namespace sv

extern "C" {

int sv_evp_create(const sv_evp_cfg* cfg, sv_evp_handle** out) {
  using namespace sv;
  SV_CHECK(cfg && out, "null argument");
  for (int s = 0; s < 4; ++s) {
    SV_CHECK(cfg->embed_dims[s] > 0 && cfg->num_heads[s] > 0 && cfg->depths[s] > 0 && cfg->sr_ratios[s] > 0, "evp: non-positive config entry");
    SV_CHECK(cfg->embed_dims[s] % 32 == 0, "evp: embed_dims must be multiples of 32 (adapter width C/4 must be a multiple of 8)");
    SV_CHECK(cfg->embed_dims[s] % cfg->num_heads[s] == 0, "evp: dim not divisible by heads");
    SV_CHECK(cfg->embed_dims[s] <= 512, "evp: embed_dims up to 512 are supported");
    const int hd = cfg->embed_dims[s] / cfg->num_heads[s];
    if (hd != 32 && hd != 64) return fail(SV_ERR_UNSUPPORTED, "evp: block attention head_dim must be 32 or 64");
  }
  SV_CHECK(cfg->mlp_ratio >= 1 && cfg->embedding_dim % 16 == 0 && cfg->embedding_dim > 0, "evp: mlp_ratio / embedding_dim");
  int dev = 0;
  SV_CUDA_OK(cudaGetDevice(&dev));
  sv_evp* h = new sv_evp();
  h->cfg = *cfg;
  h->device = dev;
  *out = h;
  return SV_OK;
}

int sv_evp_destroy(sv_evp_handle* h) {
  if (!h) return SV_OK;
  if (h->d_wb) cudaFree(h->d_wb);
  if (h->d_wf) cudaFree(h->d_wf);
  delete h;
  return SV_OK;
}

int sv_evp_set_tensor(sv_evp_handle* h, const char* name, const float* host_data, const int64_t* shape, int32_t ndim) {
  using namespace sv;
  SV_CHECK(h && name, "null argument");
  SV_CHECK(ndim >= 0 && ndim <= 4, "evp: tensor rank");
  return h->sd.set(name, host_data, shape, ndim);
}

int sv_evp_pack_weights(sv_evp_handle* h) {
  using namespace sv;
  SV_CHECK(h, "null handle");
  return pack_all(h);
}

size_t sv_evp_workspace_bytes(const sv_evp_handle* h, int32_t micro_batch, int32_t H, int32_t W) {
  if (!h || micro_batch <= 0 || H <= 0 || W <= 0) return 0;
  size_t bytes = 0;
  // sized for the larger of the two schedules (with the flow branch); configurations whose flow branch is unsupported can only
  // ever run without it
  if (sv::build(const_cast<sv_evp*>(h), nullptr, nullptr, micro_batch, H, W, sv::flow_supported(h->cfg), false, false, &bytes) != SV_OK) return 0;
  return bytes;
}

}  // extern "C"

namespace sv {
namespace {
// maps == nullptr: the plain forward.  Otherwise the capture plans run, and block k's maps of frames [b0, b0 + n) go to
// maps + off[k] + b0 * heads_k * N_k * Nkv_k.
// stage_out != nullptr: the encoder-only plans run (no flow, no features), and stage s of frames [b0, b0 + n) goes to
// stage_out[s] + b0 * C_s * H_s * W_s.
int evp_forward(sv_evp_handle* h, const float* x, const float* seg, const float* flow, float* out_features, float* maps, const std::vector<int64_t>& off,
                const std::vector<int32_t>& dims, float* const* stage_out, int32_t B, int32_t H, int32_t W, int32_t micro_batch, void* workspace,
                size_t workspace_bytes, void* stream) {
  SV_CHECK(h && x && seg && (out_features || stage_out) && workspace, "null argument");
  if (!h->sd.packed) return fail(SV_ERR_STATE, "evp: pack_weights() has not been called");
  SV_CHECK(B > 0 && micro_batch > 0, "evp: B and micro_batch must be positive");
  SV_CHECK((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "evp: workspace must be 256-byte aligned");
  SV_CHECK(static_cast<int64_t>(micro_batch) * H * W < (1LL << 28), "evp: micro_batch * H * W too large");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bool with_flow = flow != nullptr;
  h->launches = 0;
  const int E = h->cfg.embedding_dim;
  const bool capture = maps != nullptr;
  const bool features_only = stage_out != nullptr;
  std::vector<float*> block_maps(capture ? off.size() - 1 : 0);
  StageGeom g[4];
  if (features_only) stage_geometry(h->cfg, H, W, g);
  float* stage_ptr[4] = {nullptr, nullptr, nullptr, nullptr};
  for (int b0 = 0; b0 < B; b0 += micro_batch) {
    const int n = std::min<int>(micro_batch, B - b0);
    const long long key = (static_cast<long long>(n) << 40) ^ (static_cast<long long>(H) << 24) ^ (static_cast<long long>(W) << 8) ^ (with_flow ? 1 : 0) ^ (capture ? 2 : 0) ^
                         (features_only ? 4 : 0);
    auto it = h->plans.find(key);
    if (it == h->plans.end() || it->second->ws != workspace) {
      std::unique_ptr<Plan> p(new Plan());
      p->n = n; p->H = H; p->W = W; p->with_flow = with_flow; p->ws = workspace;
      SV_TRY(build(h, p.get(), workspace, n, H, W, with_flow, capture, features_only, &p->need));
      if (it == h->plans.end() && h->plans.size() >= kMaxPlans) {  // evict the least recently used plan (never the one just run)
        auto victim = h->plans.end();
        for (auto jt = h->plans.begin(); jt != h->plans.end(); ++jt)
          if (victim == h->plans.end() || jt->second->last_use < victim->second->last_use) victim = jt;
        if (victim->second.get() == h->last_plan) h->last_plan = nullptr;
        h->plans.erase(victim);
      }
      if (it != h->plans.end() && it->second.get() == h->last_plan) h->last_plan = nullptr;
      it = h->plans.insert_or_assign(key, std::move(p)).first;
    }
    // checked on EVERY call: a cached plan addresses `need` bytes behind `workspace`, whatever size the caller passes this time
    if (it->second->need > workspace_bytes) return fail(SV_ERR_INVALID, "evp: workspace too small for plan");
    it->second->last_use = ++h->plan_clock;
    const Plan& plan = *it->second;
    const size_t in_off = static_cast<size_t>(b0) * 3 * H * W;
    for (size_t k = 0; k < block_maps.size(); ++k)
      block_maps[k] = maps + off[k] + static_cast<int64_t>(b0) * dims[3 * k] * dims[3 * k + 1] * dims[3 * k + 2];
    if (features_only)
      for (int s = 0; s < 4; ++s) stage_ptr[s] = stage_out[s] + static_cast<int64_t>(b0) * g[s].C * g[s].N;
    const CallIO io{x + in_off, seg + in_off, with_flow ? flow + static_cast<size_t>(b0) * 2 * H * W : nullptr,
                    out_features ? out_features + static_cast<size_t>(b0) * E : nullptr, block_maps.data(), stage_ptr};
    SV_TRY(run_plan(h, plan, io, st));
    h->last_plan = it->second.get();
  }
  return SV_OK;
}
}  // namespace
}  // namespace sv

extern "C" {

int sv_evp_forward(sv_evp_handle* h, const float* x, const float* seg, const float* flow, float* out_features, int32_t B, int32_t H,
                   int32_t W, int32_t micro_batch, void* workspace, size_t workspace_bytes, void* stream) {
  return sv::evp_forward(h, x, seg, flow, out_features, nullptr, {}, {}, nullptr, B, H, W, micro_batch, workspace, workspace_bytes, stream);
}

int sv_evp_attention_maps_layout(const sv_evp_cfg* cfg, int32_t B, int32_t H, int32_t W, int64_t* block_offsets, int32_t* block_dims,
                                 int32_t max_blocks, int32_t* n_blocks) {
  using namespace sv;
  SV_CHECK(cfg && n_blocks, "null argument");
  std::vector<int64_t> off;
  std::vector<int32_t> dims;
  SV_TRY(maps_layout(*cfg, B, H, W, &off, &dims));
  const int nb = static_cast<int>(off.size()) - 1;
  *n_blocks = nb;
  if (!block_offsets && !block_dims) return SV_OK;  // size query
  SV_CHECK(block_offsets && block_dims, "evp: block_offsets and block_dims must both be given (or both NULL to query n_blocks)");
  SV_CHECK(max_blocks >= nb, "evp: max_blocks is smaller than n_blocks = sum(depths)");
  std::copy(off.begin(), off.end(), block_offsets);
  std::copy(dims.begin(), dims.end(), block_dims);
  return SV_OK;
}

int sv_evp_forward_attention(sv_evp_handle* h, const float* x, const float* seg, const float* flow, float* out_features, float* maps,
                             int64_t maps_elems, int32_t B, int32_t H, int32_t W, int32_t micro_batch, void* workspace, size_t workspace_bytes,
                             void* stream) {
  using namespace sv;
  SV_CHECK(h && maps, "null argument");
  std::vector<int64_t> off;
  std::vector<int32_t> dims;
  SV_TRY(maps_layout(h->cfg, B, H, W, &off, &dims));
  SV_CHECK((reinterpret_cast<uintptr_t>(maps) & 15) == 0, "evp: maps must be 16-byte aligned");
  if (maps_elems < off.back())
    return fail(SV_ERR_INVALID, "evp: maps buffer too small: " + std::to_string(maps_elems) + " elements given, " + std::to_string(off.back()) +
                                    " needed (sv_evp_attention_maps_layout)");
  return evp_forward(h, x, seg, flow, out_features, maps, off, dims, nullptr, B, H, W, micro_batch, workspace, workspace_bytes, stream);
}

int sv_evp_stage_shapes(const sv_evp_cfg* cfg, int32_t H, int32_t W, int32_t dims[12]) {
  using namespace sv;
  SV_CHECK(cfg && dims, "null argument");
  StageGeom g[4];
  SV_TRY(features_pyramid(*cfg, H, W, g));
  for (int s = 0; s < 4; ++s) {
    dims[3 * s] = g[s].C;
    dims[3 * s + 1] = g[s].H;
    dims[3 * s + 2] = g[s].W;
  }
  return SV_OK;
}

int sv_evp_forward_features(sv_evp_handle* h, const float* x, const float* seg, float* const stage_out[4], const int64_t stage_elems[4],
                            float* maps, int64_t maps_elems, int32_t B, int32_t H, int32_t W, int32_t micro_batch, void* workspace,
                            size_t workspace_bytes, void* stream) {
  using namespace sv;
  SV_CHECK(h && x && seg && stage_out && stage_elems && workspace, "null argument");
  SV_CHECK(B > 0 && micro_batch > 0, "evp: B and micro_batch must be positive");
  StageGeom g[4];
  SV_TRY(features_pyramid(h->cfg, H, W, g));
  for (int s = 0; s < 4; ++s) {
    const std::string what = "evp: stage_out[" + std::to_string(s) + "]";
    if (!stage_out[s]) return fail(SV_ERR_INVALID, what + " is NULL");
    if ((reinterpret_cast<uintptr_t>(stage_out[s]) & 3) != 0) return fail(SV_ERR_INVALID, what + " must be 4-byte aligned");
    const int64_t need = static_cast<int64_t>(B) * g[s].C * g[s].N;
    if (stage_elems[s] < need)
      return fail(SV_ERR_INVALID, what + " too small: " + std::to_string(stage_elems[s]) + " elements given, " + std::to_string(need) +
                                      " needed (B * C * H * W of sv_evp_stage_shapes)");
  }
  std::vector<int64_t> off;
  std::vector<int32_t> dims;
  if (maps) {
    SV_TRY(maps_layout(h->cfg, B, H, W, &off, &dims));
    SV_CHECK((reinterpret_cast<uintptr_t>(maps) & 15) == 0, "evp: maps must be 16-byte aligned");
    if (maps_elems < off.back())
      return fail(SV_ERR_INVALID, "evp: maps buffer too small: " + std::to_string(maps_elems) + " elements given, " + std::to_string(off.back()) +
                                      " needed (sv_evp_attention_maps_layout)");
  }
  return evp_forward(h, x, seg, nullptr, nullptr, maps, off, dims, stage_out, B, H, W, micro_batch, workspace, workspace_bytes, stream);
}

int sv_evp_classify(sv_evp_handle* h, const float* feats, float* y, float* y_ant, int32_t B, void* stream) {
  using namespace sv;
  SV_CHECK(h && feats && y && y_ant && B > 0, "bad argument");
  if (!h->sd.packed) return fail(SV_ERR_STATE, "evp: pack_weights() has not been called");
  SV_CHECK(h->cfg.embedding_dim == 2048, "evp: classifier heads expect 2048-d features");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* outs[2] = {y, y_ant};
  for (int a = 0; a < 2; ++a) {
    classify_kernel<<<B, 512, 0, st>>>(feats, h->d_wf + h->fc_w[a][0], h->d_wf + h->fc_b[a][0], h->d_wf + h->fc_w[a][1], h->d_wf + h->fc_b[a][1], outs[a]);
    SV_TRY(launch_status("classify_kernel"));
  }
  return SV_OK;
}

int sv_evp_read_tap(sv_evp_handle* h, const char* name, float* dst, int64_t max_elems, int64_t* n_elems, void* stream) {
  using namespace sv;
  SV_CHECK(h && name && dst, "null argument");
  if (!h->last_plan) return fail(SV_ERR_STATE, "evp: no forward has run yet");
  auto it = h->last_plan->taps.find(name);
  if (it == h->last_plan->taps.end()) return fail(SV_ERR_INVALID, std::string("evp: unknown tap '") + name + "'");
  if (n_elems) *n_elems = it->second.elems;
  SV_CHECK(it->second.elems <= max_elems, "evp: tap destination too small");
  return launch_bf16_to_f32(it->second.ptr, dst, it->second.elems, static_cast<cudaStream_t>(stream));
}

int64_t sv_evp_last_launch_count(const sv_evp_handle* h) { return h ? h->launches : 0; }

int sv_evp_set_profile(sv_evp_handle* h, int32_t enable) {
  using namespace sv;
  SV_CHECK(h, "null handle");
  h->profile = enable != 0;
  for (int i = 0; i < OP_KINDS; ++i) { h->prof_ms[i] = 0.0; h->prof_n[i] = 0; h->prof_bytes[i] = 0.0; }
  h->prof_gemm_flops = 0.0;
  for (auto& kv : h->plans)
    for (const Op& op : kv.second->ops) { op.prof_ms = 0.0; op.prof_n = 0; }
  return SV_OK;
}

int sv_evp_dump_profile(const sv_evp_handle* h, const char* path) {
  using namespace sv;
  SV_CHECK(h && path, "null argument");
  FILE* f = fopen(path, "w");
  if (!f) return fail(SV_ERR_INVALID, std::string("cannot open ") + path);
  static const char* kinds[] = {"gemm", "layernorm", "im2col", "dwconv", "attention", "gauss", "bilinear", "mean", "stem"};
  fprintf(f, "plan_n,op,kind,M,N,K,block_n,stages,grid,act,out_fp32,resid,i0,i1,i2,i3,i4,calls,ms_total\n");
  for (const auto& kv : h->plans) {
    const Plan& p = *kv.second;
    for (size_t i = 0; i < p.ops.size(); ++i) {
      const Op& op = p.ops[i];
      if (op.prof_n == 0) continue;
      std::visit([&](const auto& r) {
        if constexpr (std::is_same_v<std::decay_t<decltype(r)>, GemmOp>) {
          const GemmParams& g = r.plan.p;
          fprintf(f, "%d,%zu,%s,%d,%d,%d,%d,%d,%d,%d,%d,%d,0,0,0,0,0,%lld,%.6f\n", p.n, i, kinds[r.kind], g.M, g.N, g.K, g.block_n, g.num_stages,
                  r.plan.grid, g.act, g.out_fp32, g.residual != nullptr, op.prof_n, op.prof_ms);
        } else {
          const ProfCols c = r.cols();
          fprintf(f, "%d,%zu,%s,%lld,0,0,0,0,0,0,0,0,%d,%d,%d,%d,%d,%lld,%.6f\n", p.n, i, kinds[r.kind], c.M, c.i[0], c.i[1], c.i[2], c.i[3], c.i[4],
                  op.prof_n, op.prof_ms);
        }
      }, op.rec);
    }
  }
  fclose(f);
  return SV_OK;
}

int sv_evp_get_profile(const sv_evp_handle* h, double* ms_by_kind, int64_t* launches_by_kind, double* gemm_flops, double* bytes_by_kind) {
  using namespace sv;
  SV_CHECK(h && ms_by_kind && launches_by_kind && gemm_flops, "null argument");
  for (int i = 0; i < OP_KINDS; ++i) {
    ms_by_kind[i] = h->prof_ms[i];
    launches_by_kind[i] = h->prof_n[i];
    if (bytes_by_kind) bytes_by_kind[i] = h->prof_bytes[i];
  }
  *gemm_flops = h->prof_gemm_flops;
  return SV_OK;
}

}  // extern "C"
