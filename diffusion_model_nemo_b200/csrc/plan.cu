// plan.cu -- the U-Net "plan": parameter table + weight packing + the static launch program of one
// Unet.forward (modules/unet.py:131-168), the CUDA-graph loop driver and the C ABI around them.
//
// The launch program is built once from dmn_unet_cfg by mirroring Unet.__init__ (modules/unet.py:43-120):
//   init_conv -> [ResnetBlock, ResnetBlock, Residual(PreNorm(LinearAttention)), Downsample] x levels
//             -> ResnetBlock, Residual(PreNorm(Attention)), ResnetBlock
//             -> [cat skip, ResnetBlock, ResnetBlock, Residual(PreNorm(LinearAttention)), Upsample] x (levels-1)
//             -> ResnetBlock, GroupNorm, SiLU, Conv1x1
// Fusion map (what each launch covers):
//   conv (block1.proj)            : + bias, + GroupNorm statistics of its output
//   conv (block2.proj)            : prologue = GroupNorm-apply(block1.norm) + SiLU + time-embedding add on the
//                                   operand load; + bias, + statistics
//   gn_finalize                   : SiLU(GroupNorm(block2)) + residual  (+ statistics for the following PreNorm)
//   conv 1x1 (to_qkv)             : prologue = PreNorm GroupNorm(1) apply
//   linattn_core / attn_core      : both softmaxes, scale and the two small contractions
//   conv 1x1 (to_out)             : + bias (+ statistics of GroupNorm(1) | + residual for the bottleneck Attention)
//   gn_finalize                   : GroupNorm(1) + residual
//   concat                        : never materialised (two-source operand load)
#include <cfloat>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "../../include/dmn_b200.h"
#include "common.cuh"
#include "ops.h"

namespace dmn {

static thread_local std::string g_err;
thread_local long g_launches = 0;
void set_error(const std::string& m) { g_err = m; }
bool pdl_enabled() {
  static const bool on = [] {
    const char* e = getenv("DMN_PDL");
    return e && e[0] == '1';      // opt-in: measured neutral inside the CUDA graph (profiles/README.md)
  }();
  return on;
}
int fail(int code, const std::string& m) {
  g_err = m;
  return code;
}

int launch_advance_counter(int32_t* c, cudaStream_t st);
int launch_set_counter(int32_t* c, int v, dmn_rng rng, cudaStream_t st);
int launch_ddpm(const float* x, const float* eps, const float* z, float* out, long n, const float* coef, const int32_t* step_dev,
                int step, dmn_rng rng, const dmn_rng* rng_dev, cudaStream_t st);
int launch_learned(const float* x, const float* mo, const float* z, float* out, int batch, long chw, const float* coef,
                   const int32_t* step_dev, int step, dmn_rng rng, const dmn_rng* rng_dev, cudaStream_t st);
int launch_ddim(const float* x, const float* eps, const float* z, float* out, long n, const float* coef, const int32_t* step_dev,
                int step, dmn_rng rng, const dmn_rng* rng_dev, cudaStream_t st);
int launch_dpmpp(const float* x, const float* mo, float* hist, float* out, int batch, long chw, long mo_chw, const float* coef,
                 const float* coef2, const float* z, const int32_t* step_dev, int step, dmn_rng rng, const dmn_rng* rng_dev, cudaStream_t st);
int launch_inpaint_prepare(const float* x, const float* known, const float* mask, float* out, long n, const float* coef,
                           const int32_t* step_dev, int step, dmn_rng rng, const dmn_rng* rng_dev, cudaStream_t st);
int launch_traj(const float* x, float* traj, long n, const int32_t* step_dev, int every, int n_steps, cudaStream_t st);
int launch_bpd_qsample(const float* x0, const float* z, float* xt, long n, const float* coef, const int32_t* step_dev, int step, dmn_rng rng,
                       const dmn_rng* rng_dev, cudaStream_t st);
int launch_bpd_term(const float* x0, const float* xt, const float* mo, float* terms, int batch, long chw, int learned, int n_cols, int mode,
                    const float* coef, const float* coef2, const int32_t* step_dev, int step, cudaStream_t st);
int launch_cfg_dup(const float* x, float* x2, long n, cudaStream_t st);
int launch_cfg_combine(const float* mo2, float* mo, long n, long per_sample, long guided, float w, cudaStream_t st);
int launch_langevin(const float* x, const float* mo, const float* z, float* out, float* mean_out, int batch, long chw,
                    float snr, const float* coef, const int32_t* step_dev, int step, int draw, float* scratch, dmn_rng rng,
                    const dmn_rng* rng_dev, cudaStream_t st);
int launch_affine_noise(const float* x, const float* mo, const float* z, float* out, float* mean_out, long n, const float* coef,
                        const int32_t* step_dev, int step, int draw, dmn_rng rng, const dmn_rng* rng_dev, cudaStream_t st);

enum ParamKind {
  PK_RAW,        // copied as is (bias, gamma, beta, final 1x1 weight, class embedding)
  PK_CONV,       // convolution weight -> engine layout(s)
  PK_INIT,       // init_conv weight [dim][ch][7][7] -> [49*ch][dim]
  PK_LIN_T,      // Linear weight [out][in] -> [in][out]
  PK_BLOCK_MLP_W,  // ResnetBlock.mlp.1.weight [cout][4dim] -> column slice of [4dim][sumC]
  PK_BLOCK_MLP_B,  // ResnetBlock.mlp.1.bias -> slice of [sumC]
  PK_PLAIN_BF16,   // 1x1 conv weight [out][in][1][1] -> row-major bf16 [out][in] (TMA operand of the fused attention kernel)
};

struct Param {
  std::string name;
  std::vector<int64_t> shape;
  int kind = PK_RAW;
  size_t off = 0;        // primary device region (bytes from weights base)
  size_t off2 = 0;       // PK_CONV: tcgen05 image (0 = none)
  bool has_simt = true;  // PK_CONV: SIMT image present
  bool has_tc = false;   // PK_CONV: tcgen05 image present
  int mode = 0, ksize = 0, cin = 0, cout = 0;   // PK_CONV
  int col = 0;           // PK_BLOCK_MLP_*: column offset
  bool loaded = false;
  bool keep_host = false;          // parameters of a folded to_qkv: host copy kept until all three (weight, gamma, beta) arrived
  int fold_op = -1;                // op index of that conv
  std::vector<float> host;
  int64_t numel() const {
    int64_t n = 1;
    for (auto s : shape) n *= s;
    return n;
  }
};

enum OpKind { OP_MEMSET, OP_INIT, OP_CONV, OP_FINALIZE, OP_LINATTN, OP_ATTN, OP_FINALPROJ, OP_MODULATE, OP_CLASSADD, OP_ATTN_FUSED };

// Buffers are addressed as (region id, so pointers can be resolved after bind)
struct Buf {
  size_t off = (size_t)-1;   // bytes from workspace base
  bool valid() const { return off != (size_t)-1; }
};

struct Op {
  int kind = OP_CONV;
  std::string name;
  // conv
  int mode = 0, ksize = 3, C1 = 0, C2 = 0, Cout = 0, Hin = 0, Hout = 0;
  Buf src1, src2, out, res;
  int w = -1, bias = -1;            // param indices
  int pro = 0, pgroups = 0, pgamma = -1, pbeta = -1;
  Buf pstats, ostats;
  int ogroups = 0;
  int temb_col = -1;
  bool tc = false;                  // tcgen05 engine for this conv
  // to_qkv with the PreNorm GroupNorm(1) folded into weights + epilogue affine (ops.h: ConvP::fold_s1)
  bool fold = false;
  int fold_gamma = -1, fold_beta = -1;
  size_t fold_off = 0;              // s1 | s2, 2 * Cout floats in the weight arena
  // finalize / final proj
  int groups = 0, gamma = -1, beta = -1, silu = 0, C = 0, HW = 0;
  Buf raw, stats;
  // attention
  int heads = 4, dh = 32, N = 0;
  int wo = -1, bo = -1;             // fused attention block: to_out.0 weight (plain bf16 image) / bias
  bool softmax = false;             // fused attention block: the bottleneck softmax Attention instead of LinearAttention
};

}  // namespace dmn

using namespace dmn;

struct dmn_plan {
  dmn_unet_cfg cfg;
  int act = 0, engine = 0;
  size_t esz = 4;
  std::vector<Param> params;
  std::map<std::string, int> pidx;
  std::vector<Op> ops;
  size_t weights_bytes = 0, ws_bytes = 0;
  char* wbase = nullptr;
  char* wsbase = nullptr;
  // time path
  int sumC = 0;
  size_t off_freqs = 0, off_wct = 0, off_bc = 0;
  bool freqs_loaded = false;
  // FiLM (WaveGradUNet): channels of every evaluated FiLM layer, in table-column order
  std::vector<int> film_channels, film_cols;   // film_cols: first table column of each FiLM layer
  Buf time_tmp, time_table;
  // statistics arena
  size_t stats_off = 0, stats_bytes = 0;
  Buf out_nhwc_dummy;
  int launches_per_forward = 0;
  bool init_tc = false;            // stem on the tensor-core engine
  // loop state
  Buf counters;   // int32[4]
  struct GraphEntry {
    cudaGraphExec_t exec = nullptr;
    dmn_loop_desc key;
    dmn_inpaint_desc ip{};   // all null for a plain sampling loop
  };
  std::vector<GraphEntry> graphs;
  template <class Desc>
  struct OdeGraphEntry {
    cudaGraphExec_t exec = nullptr;
    Desc key;
  };
  std::vector<OdeGraphEntry<dmn_ode_desc>> ode_graphs;
  std::vector<OdeGraphEntry<dmn_ode_likelihood_desc>> lik_graphs;
  void drop_graphs() {
    for (auto& g : graphs)
      if (g.exec) cudaGraphExecDestroy(g.exec);
    graphs.clear();
    for (auto& g : ode_graphs)
      if (g.exec) cudaGraphExecDestroy(g.exec);
    ode_graphs.clear();
    for (auto& g : lik_graphs)
      if (g.exec) cudaGraphExecDestroy(g.exec);
    lik_graphs.clear();
  }
  ~dmn_plan() { drop_graphs(); }
};

namespace dmn {

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct Builder {
  dmn_plan& P;
  size_t woff = 0, wsoff = 0;
  explicit Builder(dmn_plan& p) : P(p) {}

  size_t walloc(size_t bytes) {
    size_t o = woff;
    woff = align_up(woff + bytes, 256);
    return o;
  }
  Buf wsalloc(size_t bytes) {
    Buf b;
    b.off = wsoff;
    wsoff = align_up(wsoff + bytes, 256);
    return b;
  }
  Buf act(int HW, int C) { return wsalloc((size_t)P.cfg.max_batch * HW * C * P.esz); }
  Buf stats(int G) {
    Buf b;
    b.off = P.stats_off + P.stats_bytes;
    P.stats_bytes += align_up((size_t)P.cfg.max_batch * G * 2 * sizeof(stat_t), 256);
    return b;
  }

  int add_param(const std::string& name, std::vector<int64_t> shape, int kind) {
    Param q;
    q.name = name;
    q.shape = std::move(shape);
    q.kind = kind;
    if (kind == PK_RAW || kind == PK_INIT || kind == PK_LIN_T) q.off = walloc((size_t)q.numel() * sizeof(float));
    P.params.push_back(q);
    P.pidx[name] = (int)P.params.size() - 1;
    return (int)P.params.size() - 1;
  }
  int add_conv_param(const std::string& name, int mode, int ksize, int cin, int cout, bool tc) {
    Param q;
    q.name = name;
    const int k = (mode == CONV_SAME) ? ksize : 4;
    if (mode == CONV_UP) q.shape = {cin, cout, k, k};
    else q.shape = {cout, cin, k, k};
    q.kind = PK_CONV;
    q.mode = mode; q.ksize = ksize; q.cin = cin; q.cout = cout;
    q.has_simt = !tc;
    if (q.has_simt) q.off = walloc((size_t)q.numel() * sizeof(float));
    q.has_tc = tc;
    if (tc) q.off2 = walloc(conv_tcgen05_weight_bytes(mode, ksize, cin, cout));
    P.params.push_back(q);
    P.pidx[name] = (int)P.params.size() - 1;
    return (int)P.params.size() - 1;
  }

  int add_plain_param(const std::string& name, int cout, int cin) {
    Param q;
    q.name = name;
    q.shape = {cout, cin, 1, 1};
    q.kind = PK_PLAIN_BF16;
    q.cin = cin; q.cout = cout;
    q.off = walloc((size_t)cout * cin * 2);
    P.params.push_back(q);
    P.pidx[name] = (int)P.params.size() - 1;
    return (int)P.params.size() - 1;
  }

  bool want_tc(int mode, int ksize, int C1, int C2, int Cout, int Hin, int pro, int pgroups, int ogroups) {
    if (P.engine != DMN_CONV_TCGEN05) return false;
    ConvP c;
    c.mode = mode; c.ksize = ksize; c.C1 = C1; c.C2 = C2; c.Cout = Cout;
    c.B = P.cfg.max_batch; c.Hin = c.Win = Hin;
    c.Hout = c.Wout = (mode == CONV_DOWN) ? Hin / 2 : (mode == CONV_UP ? Hin * 2 : Hin);
    c.pro = pro; c.pgroups = pgroups; c.ogroups = ogroups;
    return conv_tcgen05_supported(c);
  }

  // conv op; returns op index
  int conv(const std::string& pname, int mode, int ksize, Buf s1, int C1, Buf s2, int C2, int Cout, int Hin, Buf out,
           bool has_bias, int ogroups, int pro = 0, int pgroups = 0, Buf pstats = Buf(), int pgamma = -1, int pbeta = -1,
           int temb_col = -1, Buf res = Buf()) {
    Op o;
    o.kind = OP_CONV;
    o.name = pname;
    o.mode = mode; o.ksize = ksize; o.C1 = C1; o.C2 = C2; o.Cout = Cout; o.Hin = Hin;
    o.Hout = (mode == CONV_DOWN) ? Hin / 2 : (mode == CONV_UP ? Hin * 2 : Hin);
    o.src1 = s1; o.src2 = s2; o.out = out; o.res = res;
    o.tc = want_tc(mode, ksize, C1, C2, Cout, Hin, pro, pgroups, ogroups);
    o.w = add_conv_param(pname + ".weight", mode, ksize, C1 + C2, Cout, o.tc);
    if (has_bias) o.bias = add_param(pname + ".bias", {Cout}, PK_RAW);
    o.pro = pro; o.pgroups = pgroups; o.pstats = pstats; o.pgamma = pgamma; o.pbeta = pbeta; o.temb_col = temb_col;
    o.ogroups = ogroups;
    if (ogroups > 0) o.ostats = stats(ogroups);
    P.ops.push_back(o);
    return (int)P.ops.size() - 1;
  }

  // ResnetBlock (parts/convnext.py:63-86).  x_in: (s1,C1)+(s2,C2) -> out (Cout channels)
  void resblock(const std::string& p, Buf s1, int C1, Buf s2, int C2, int Cout, int H, Buf h1, Buf h2, Buf rbuf, Buf out,
                bool temb, int ostats_groups, Buf* ostats_out) {
    const int G = P.cfg.groups;
    const int Cin = C1 + C2;
    int temb_col = -1;
    if (temb && P.cfg.with_time_emb) {
      temb_col = P.sumC;
      Param w; w.name = p + ".mlp.1.weight"; w.shape = {Cout, 4 * P.cfg.dim}; w.kind = PK_BLOCK_MLP_W; w.col = temb_col;
      P.params.push_back(w); P.pidx[w.name] = (int)P.params.size() - 1;
      Param b; b.name = p + ".mlp.1.bias"; b.shape = {Cout}; b.kind = PK_BLOCK_MLP_B; b.col = temb_col;
      P.params.push_back(b); P.pidx[b.name] = (int)P.params.size() - 1;
      P.sumC += Cout;
    }
    // block1: conv -> (GroupNorm, SiLU deferred to the consumer)
    int c1 = conv(p + ".block1.proj", CONV_SAME, 3, s1, C1, s2, C2, Cout, H, h1, true, G);
    int g1w = add_param(p + ".block1.norm.weight", {Cout}, PK_RAW);
    int g1b = add_param(p + ".block1.norm.bias", {Cout}, PK_RAW);
    Buf res = s1;
    if (Cin != Cout) {
      conv(p + ".res_conv", CONV_SAME, 1, s1, C1, s2, C2, Cout, H, rbuf, true, 0);
      res = rbuf;
    }
    // block2: conv( SiLU(GN(h1)) + temb )
    int pro = PRO_GN | PRO_SILU | (temb_col >= 0 ? PRO_TEMB : 0);
    int c2 = conv(p + ".block2.proj", CONV_SAME, 3, h1, Cout, Buf(), 0, Cout, H, h2, true, G, pro, G, P.ops[c1].ostats, g1w, g1b,
                  temb_col);
    int g2w = add_param(p + ".block2.norm.weight", {Cout}, PK_RAW);
    int g2b = add_param(p + ".block2.norm.bias", {Cout}, PK_RAW);
    Op f;
    f.kind = OP_FINALIZE;
    f.name = p + ".finalize";
    f.raw = h2; f.stats = P.ops[c2].ostats; f.groups = G; f.gamma = g2w; f.beta = g2b; f.silu = 1;
    f.res = res; f.out = out; f.C = Cout; f.HW = H * H;
    f.ogroups = ostats_groups;
    if (ostats_groups > 0) {
      f.ostats = stats(ostats_groups);
      if (ostats_out) *ostats_out = f.ostats;
    }
    P.ops.push_back(f);
  }

  // FeatureWiseLinearModulation (parts/film.py:29-61): signal conv3x3 -> [LeakyReLU(0.2) + positional encoding of the noise level,
  // fused into the operand load of the next two convs] -> scale conv3x3, shift conv3x3
  void film(int idx, Buf x, int C, int H, Buf tmp, Buf scale, Buf shift) {
    const std::string p = "films." + std::to_string(idx);
    const int col = P.sumC;
    P.sumC += C;
    P.film_channels.push_back(C);
    P.film_cols.push_back(col);
    conv(p + ".signal_conv.0", CONV_SAME, 3, x, C, Buf(), 0, C, H, tmp, true, 0);
    conv(p + ".scale_conv", CONV_SAME, 3, tmp, C, Buf(), 0, C, H, scale, true, 0, PRO_LRELU | PRO_TEMB, 0, Buf(), -1, -1, col);
    conv(p + ".shift_conv", CONV_SAME, 3, tmp, C, Buf(), 0, C, H, shift, true, 0, PRO_LRELU | PRO_TEMB, 0, Buf(), -1, -1, col);
  }
  // x = x * scale + shift   (modules/unet.py:259,262)
  void modulate(const std::string& name, Buf x, Buf scale, Buf shift, int C, int H) {
    Op m;
    m.kind = OP_MODULATE;
    m.name = name;
    m.src1 = x; m.src2 = scale; m.res = shift; m.out = x; m.C = C; m.HW = H * H;
    P.ops.push_back(m);
  }

  // Residual(PreNorm(dim, LinearAttention | Attention))   (utils.py:68-93, parts/mha.py)
  void attn_block(const std::string& p, bool linear, Buf x, Buf xstats, int C, int H, Buf qkv, Buf att, Buf oraw, Buf out) {
    const int hidden = 128;
    int nw = add_param(p + ".fn.norm.weight", {C}, PK_RAW);
    int nb = add_param(p + ".fn.norm.bias", {C}, PK_RAW);
    static const bool no_fused = [] { const char* e = getenv("DMN_NO_FUSED_ATTN"); return e && e[0] == '1'; }();
    if (linear && !no_fused && P.engine == DMN_CONV_TCGEN05 && linattn_fused_supported(P.cfg.max_batch, H * H, C)) {
      // the whole Residual(PreNorm(LinearAttention)) block as one tcgen05 kernel (attn_fused.cu): q / k / v never reach global memory
      Op a;
      a.kind = OP_ATTN_FUSED;
      a.name = p + ".fused";
      a.src1 = x; a.out = out; a.pstats = xstats; a.C = C; a.N = H * H; a.HW = H * H; a.Hin = H;
      a.w = add_plain_param(p + ".fn.fn.to_qkv.weight", 3 * hidden, C);
      a.fold = true;
      a.fold_gamma = nw;
      a.fold_beta = nb;
      a.fold_off = walloc((size_t)2 * 3 * hidden * sizeof(float));
      a.wo = add_plain_param(p + ".fn.fn.to_out.0.weight", C, hidden);
      a.bo = add_param(p + ".fn.fn.to_out.0.bias", {C}, PK_RAW);
      a.gamma = add_param(p + ".fn.fn.to_out.1.weight", {C}, PK_RAW);
      a.beta = add_param(p + ".fn.fn.to_out.1.bias", {C}, PK_RAW);
      P.ops.push_back(a);
      const int ci = (int)P.ops.size() - 1;
      for (int pi : {a.w, nw, nb}) {
        P.params[pi].keep_host = true;
        P.params[pi].fold_op = ci;
      }
      return;
    }
    if (!linear && !no_fused && P.engine == DMN_CONV_TCGEN05 && attn_softmax_fused_supported(P.cfg.max_batch, H * H, C)) {
      // Residual(PreNorm(Attention)) (the bottleneck softmax attention) as one tcgen05 kernel
      Op a;
      a.kind = OP_ATTN_FUSED;
      a.name = p + ".fused";
      a.softmax = true;
      a.src1 = x; a.out = out; a.pstats = xstats; a.C = C; a.N = H * H; a.HW = H * H; a.Hin = H;
      a.w = add_plain_param(p + ".fn.fn.to_qkv.weight", 3 * hidden, C);
      a.fold = true;
      a.fold_gamma = nw;
      a.fold_beta = nb;
      a.fold_off = walloc((size_t)2 * 3 * hidden * sizeof(float));
      a.wo = add_plain_param(p + ".fn.fn.to_out.weight", C, hidden);
      a.bo = add_param(p + ".fn.fn.to_out.bias", {C}, PK_RAW);
      P.ops.push_back(a);
      const int ci = (int)P.ops.size() - 1;
      for (int pi : {a.w, nw, nb}) {
        P.params[pi].keep_host = true;
        P.params[pi].fold_op = ci;
      }
      return;
    }
    if (P.engine == DMN_CONV_TCGEN05 && want_tc(CONV_SAME, 1, C, 0, 3 * hidden, H, 0, 0, 0)) {
      // tensor-core engine: GroupNorm(1) folded through the 1x1 conv (raw operand load, affine in the epilogue)
      const int ci = conv(p + ".fn.fn.to_qkv", CONV_SAME, 1, x, C, Buf(), 0, 3 * hidden, H, qkv, false, 0);
      Op& o = P.ops[ci];
      o.fold = true;
      o.pstats = xstats;
      o.pgroups = 1;
      o.fold_gamma = nw;
      o.fold_beta = nb;
      o.fold_off = walloc((size_t)2 * 3 * hidden * sizeof(float));
      for (int pi : {o.w, nw, nb}) {
        P.params[pi].keep_host = true;
        P.params[pi].fold_op = ci;
      }
    } else {
      conv(p + ".fn.fn.to_qkv", CONV_SAME, 1, x, C, Buf(), 0, 3 * hidden, H, qkv, false, 0, PRO_GN, 1, xstats, nw, nb);
    }
    Op a;
    a.kind = linear ? OP_LINATTN : OP_ATTN;
    a.name = p + ".core";
    a.src1 = qkv; a.out = att; a.N = H * H; a.heads = 4; a.dh = 32;
    P.ops.push_back(a);
    if (linear) {
      int co = conv(p + ".fn.fn.to_out.0", CONV_SAME, 1, att, hidden, Buf(), 0, C, H, oraw, true, 1);
      int gw = add_param(p + ".fn.fn.to_out.1.weight", {C}, PK_RAW);
      int gb = add_param(p + ".fn.fn.to_out.1.bias", {C}, PK_RAW);
      Op f;
      f.kind = OP_FINALIZE;
      f.name = p + ".finalize";
      f.raw = oraw; f.stats = P.ops[co].ostats; f.groups = 1; f.gamma = gw; f.beta = gb; f.silu = 0;
      f.res = x; f.out = out; f.C = C; f.HW = H * H;
      P.ops.push_back(f);
    } else {
      conv(p + ".fn.fn.to_out", CONV_SAME, 1, att, hidden, Buf(), 0, C, H, out, true, 0, 0, 0, Buf(), -1, -1, -1, x);
    }
  }

  int build() {
    const dmn_unet_cfg& c = P.cfg;
    const int dim = c.dim, n = c.n_mults, S = c.image_size, G = c.groups;
    std::vector<int> dims = {dim};
    for (int i = 0; i < n; ++i) dims.push_back(dim * c.dim_mults[i]);
    // resolution of each level
    std::vector<int> Hs(n);
    int H = S;
    for (int i = 0; i < n; ++i) {
      Hs[i] = H;
      if (i < n - 1) {
        if (H % 2) return fail(DMN_EINVAL, "image_size must be divisible by 2^(levels-1)");
        H /= 2;
      }
    }
    // max per-sample activation size
    size_t maxact = 0, maxqkv = 0, maxatt = 0;
    for (int i = 0; i < n; ++i) {
      size_t hw = (size_t)Hs[i] * Hs[i];
      maxact = std::max(maxact, hw * std::max(dims[i], dims[i + 1]));
      maxqkv = std::max(maxqkv, hw * 384);
      maxatt = std::max(maxatt, hw * 128);
    }
    maxact = std::max(maxact, (size_t)S * S * dim);
    auto actbuf = [&](size_t per_sample) { return wsalloc((size_t)c.max_batch * per_sample * P.esz); };

    // statistics arena first (fixed offset); its size is known only after the program is built, so reserve generously
    P.stats_off = wsoff;
    const size_t stats_reserve = align_up((size_t)c.max_batch * 64 * 2 * sizeof(stat_t), 256) * 160;
    wsoff += stats_reserve;

    Buf X[3] = {actbuf(maxact), actbuf(maxact), actbuf(maxact)};
    Buf H1 = actbuf(maxact), H2 = actbuf(maxact), R = actbuf(maxact), O = actbuf(maxact);
    Buf QKV = actbuf(maxqkv), ATT = actbuf(maxatt);
    std::vector<Buf> skip(n);
    for (int i = 0; i < n; ++i) skip[i] = actbuf((size_t)Hs[i] * Hs[i] * dims[i + 1]);
    // WaveGradUNet (unet.py:204-266): FiLM 0 on the stem output, FiLM i+1 on the output of down level i; the last level's FiLM is
    // computed and discarded by the reference (unet.py:247), so it is not evaluated here.  (scale, shift) live until the up path.
    const bool film_on = c.film != 0;
    if (film_on && c.with_time_emb) return fail(DMN_EINVAL, "film requires with_time_emb = 0 (unet.py:195)");
    std::vector<Buf> fscale(n), fshift(n);
    if (film_on)
      for (int i = 0; i < n; ++i) {
        const size_t per = (size_t)Hs[i == 0 ? 0 : i - 1] * Hs[i == 0 ? 0 : i - 1] * dims[i];
        fscale[i] = actbuf(per);
        fshift[i] = actbuf(per);
      }

    // parameters that are not attached to a conv op
    {
      const int pi = add_param("init_conv.weight", {dim, c.channels, 7, 7}, PK_INIT);
      P.init_tc = P.engine == DMN_CONV_TCGEN05 && init_conv_tcgen05_supported(c.channels, S, dim, c.max_batch);
      if (P.init_tc) {
        P.params[pi].has_tc = true;
        P.params[pi].off2 = walloc(init_conv_tcgen05_weight_bytes(dim));
      }
    }
    add_param("init_conv.bias", {dim}, PK_RAW);
    if (c.with_time_emb) {
      add_param("time_mlp.1.weight", {4 * dim, dim}, PK_LIN_T);
      add_param("time_mlp.1.bias", {4 * dim}, PK_RAW);
      add_param("time_mlp.3.weight", {4 * dim, 4 * dim}, PK_LIN_T);
      add_param("time_mlp.3.bias", {4 * dim}, PK_RAW);
    }
    if (c.num_classes >= 0) add_param("class_embed.weight", {c.num_classes + 1, dim}, PK_RAW);

    Op m;
    m.kind = OP_MEMSET;
    m.name = "zero_stats";
    P.ops.push_back(m);
    Op ic;
    ic.kind = OP_INIT;
    ic.name = "init_conv";
    ic.out = X[0];
    P.ops.push_back(ic);

    int cur = 0;   // index of the X buffer holding the current activation
    Buf x = X[0];
    if (film_on) {
      film(0, x, dim, S, H1, fscale[0], fshift[0]);
      if (c.num_classes >= 0) {
        // WaveGradUNet adds the class embedding AFTER FiLM 0 has read the stem output (unet.py:214-226), so the stem runs without it
        Op a;
        a.kind = OP_CLASSADD;
        a.name = "class_embed.add";
        a.src1 = x; a.out = x; a.C = dim; a.HW = S * S;
        P.ops.push_back(a);
      }
    }
    for (int i = 0; i < n; ++i) {
      const int ci = dims[i], co = dims[i + 1], Hh = Hs[i];
      const std::string p = "downs." + std::to_string(i);
      Buf o1 = X[(cur + 1) % 3];
      resblock(p + ".0", x, ci, Buf(), 0, co, Hh, H1, H2, R, o1, true, 0, nullptr);
      Buf o2 = X[(cur + 2) % 3];
      Buf st;
      resblock(p + ".1", o1, co, Buf(), 0, co, Hh, H1, H2, R, o2, true, 1, &st);
      attn_block(p + ".2", true, o2, st, co, Hh, QKV, ATT, O, skip[i]);
      if (film_on && i < n - 1) film(i + 1, skip[i], co, Hh, H1, fscale[i + 1], fshift[i + 1]);
      if (i < n - 1) {
        Buf o3 = X[cur % 3];
        conv(p + ".3", CONV_DOWN, 4, skip[i], co, Buf(), 0, co, Hh, o3, true, 0);
        x = o3;
      } else {
        x = skip[i];
      }
    }
    const int mid = dims[n], Hm = Hs[n - 1];
    {
      Buf st;
      Buf o1 = X[(cur + 1) % 3];
      resblock("mid_block1", x, mid, Buf(), 0, mid, Hm, H1, H2, R, o1, true, 1, &st);
      Buf o2 = X[(cur + 2) % 3];
      attn_block("mid_attn", false, o1, st, mid, Hm, QKV, ATT, O, o2);
      Buf o3 = X[cur % 3];
      resblock("mid_block2", o2, mid, Buf(), 0, mid, Hm, H1, H2, R, o3, true, 0, nullptr);
      x = o3;
    }
    // ups: reversed(in_out[1:])
    int Hu = Hm;
    for (int j = 0; j < n - 1; ++j) {
      const int lvl = n - 1 - j;              // in_out[lvl] = (dims[lvl], dims[lvl+1])
      const int ci = dims[lvl], co = dims[lvl + 1];
      const std::string p = "ups." + std::to_string(j);
      // input = cat(x [co channels], skip[lvl] [co channels])
      Buf o1 = X[(cur + 1) % 3];
      resblock(p + ".0", x, co, skip[lvl], co, ci, Hu, H1, H2, R, o1, true, 0, nullptr);
      Buf o2 = X[(cur + 2) % 3];
      Buf st;
      resblock(p + ".1", o1, ci, Buf(), 0, ci, Hu, H1, H2, R, o2, true, 1, &st);
      Buf o3 = X[cur % 3];
      attn_block(p + ".2", true, o2, st, ci, Hu, QKV, ATT, O, o3);
      Buf o4 = X[(cur + 1) % 3];
      conv(p + ".3", CONV_UP, 4, o3, ci, Buf(), 0, ci, Hu, o4, true, 0);
      x = o4;
      cur = (cur + 1) % 3;
      Hu *= 2;
      if (film_on) modulate(p + ".film", x, fscale[lvl], fshift[lvl], ci, Hu);    // statistics of down level lvl-1: dims[lvl] channels at Hs[lvl-1]
    }
    if (film_on) modulate("film0", x, fscale[0], fshift[0], dim, S);
    if (Hu != S) return fail(DMN_EINVAL, "internal: resolution bookkeeping");
    // final_conv = ResnetBlock(dim, dim) without time embedding, GroupNorm, SiLU, Conv1x1
    {
      Buf st;
      Buf o1 = X[(cur + 1) % 3];
      resblock("final_conv.0", x, dim, Buf(), 0, dim, S, H1, H2, R, o1, false, c.plain_tail ? 0 : G, &st);
      Op f;
      f.kind = OP_FINALPROJ;
      f.name = "final_conv.tail";
      f.src1 = o1; f.stats = st; f.groups = G; f.C = dim; f.HW = S * S; f.Cout = c.out_dim;
      if (c.plain_tail) {          // 'conv_bn_act': the ResnetBlock is followed by the bare 1x1 (unet.py:115-116)
        f.groups = 0;
        f.w = add_param("final_conv.1.weight", {c.out_dim, dim, 1, 1}, PK_RAW);
        f.bias = add_param("final_conv.1.bias", {c.out_dim}, PK_RAW);
      } else {
        f.gamma = add_param("final_conv.1.weight", {dim}, PK_RAW);
        f.beta = add_param("final_conv.1.bias", {dim}, PK_RAW);
        f.w = add_param("final_conv.3.weight", {c.out_dim, dim, 1, 1}, PK_RAW);
        f.bias = add_param("final_conv.3.bias", {c.out_dim}, PK_RAW);
      }
      P.ops.push_back(f);
    }
    if (P.stats_bytes > stats_reserve) return fail(DMN_EINVAL, "internal: statistics arena overflow");

    // time path storage
    if (film_on) {
      P.off_freqs = walloc((size_t)2 * P.sumC * sizeof(float));     // freq | is_cos per table column
      P.time_table = wsalloc((size_t)c.max_time_rows * P.sumC * sizeof(float));
    }
    if (c.with_time_emb) {
      P.off_freqs = walloc((size_t)(dim / 2) * sizeof(float));
      P.off_wct = walloc((size_t)4 * dim * P.sumC * sizeof(float));
      P.off_bc = walloc((size_t)P.sumC * sizeof(float));
      P.time_tmp = wsalloc((size_t)c.max_time_rows * 8 * dim * sizeof(float));
      P.time_table = wsalloc((size_t)c.max_time_rows * P.sumC * sizeof(float));
    }
    P.counters = wsalloc(256);
    P.weights_bytes = woff;
    P.ws_bytes = wsoff;
    return 0;
  }
};

// DDPM loop: the final_conv tail, the posterior update and the step counter as ONE launch (sampler.cu: final_proj_ddpm_kernel)
struct TailFuse {
  const float* x = nullptr;          // x_t (also the U-Net input of this step)
  const float* z = nullptr;          // injected noise of this step or null (in-kernel Philox)
  float* out = nullptr;              // x_{t-1} (may alias x)
  const float* coef = nullptr;
  const int32_t* step_dev = nullptr;
  int step = 0;
  dmn_rng rng = {0, 0};
  const dmn_rng* rng_dev = nullptr;
  int32_t* advance = nullptr;        // loop counters when this launch also advances the step counter
};

static FinalProjP final_proj_params(const dmn_plan* P, const Op& o, float* out_dev, int batch) {
  auto W = [&](int pi) -> const float* { return pi < 0 ? nullptr : (const float*)(P->wbase + P->params[pi].off); };
  FinalProjP q;
  q.y = o.src1.valid() ? (void*)(P->wsbase + o.src1.off) : nullptr;
  q.stats = o.stats.valid() ? (const stat_t*)(P->wsbase + o.stats.off) : nullptr;
  q.groups = o.groups;
  q.gamma = W(o.gamma); q.beta = W(o.beta); q.w = W(o.w); q.bias = W(o.bias);
  q.out = out_dev; q.B = batch; q.HW = o.HW; q.C = o.C; q.Cout = o.Cout;
  q.plain = o.groups == 0;
  return q;
}

static bool tail_fusable(const dmn_plan* P) {
  static const bool off = [] { const char* e = getenv("DMN_NO_FUSED_TAIL"); return e && e[0] == '1'; }();
  if (off || P->ops.empty() || P->ops.back().kind != OP_FINALPROJ || P->cfg.out_dim != P->cfg.channels) return false;
  return fused_tail_supported(final_proj_params(P, P->ops.back(), nullptr, 1), P->act);
}

// device time stamp (nanoseconds) between the launches of a captured forward program (dmn_plan_profile_forward_graph)
__global__ void stamp_kernel(unsigned long long* t) {
  unsigned long long v;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(v));
  *t = v;
}

// one op of the forward program
static int enqueue_op(dmn_plan* P, const Op& o, const float* x_dev, const int32_t* row_dev, const int64_t* classes_dev, float* out_dev,
                      int batch, cudaStream_t st, const TailFuse* tail) {
  const dmn_unet_cfg& c = P->cfg;
  auto W = [&](int pi) -> const float* { return pi < 0 ? nullptr : (const float*)(P->wbase + P->params[pi].off); };
  auto B = [&](const Buf& b) -> void* { return b.valid() ? (void*)(P->wsbase + b.off) : nullptr; };
  int rc = 0;
  switch (o.kind) {
    case OP_MEMSET: {
      DMN_CUDA_CHECK(cudaMemsetAsync(P->wsbase + P->stats_off, 0, P->stats_bytes, st));
      count_launch();
      break;
    }
    case OP_INIT: {
      InitConvP q;
      q.x = x_dev;
      q.w = W(P->pidx["init_conv.weight"]);
      q.bias = W(P->pidx["init_conv.bias"]);
      if (c.num_classes >= 0 && !c.film) {
        q.cls_w = W(P->pidx["class_embed.weight"]);
        q.classes = classes_dev;
        q.pad_class = c.num_classes;
      }
      q.out = B(o.out);
      q.B = batch; q.Cin = c.channels; q.S = c.image_size; q.Cout = c.dim;
      if (P->init_tc) {
        q.w = (const float*)(P->wbase + P->params[P->pidx["init_conv.weight"]].off2);
        rc = init_conv_tcgen05(q, st);
      } else {
        rc = init_conv(q, P->act, st);
      }
      break;
    }
    case OP_CONV: {
      ConvP q;
      q.src1 = B(o.src1); q.src2 = B(o.src2); q.C1 = o.C1; q.C2 = o.C2;
      q.B = batch; q.Hin = q.Win = o.Hin; q.Hout = q.Wout = o.Hout; q.Cout = o.Cout;
      q.mode = o.mode; q.ksize = o.ksize;
      const Param& wp = P->params[o.w];
      q.w = o.tc ? (const void*)(P->wbase + wp.off2) : (const void*)(P->wbase + wp.off);
      q.bias = W(o.bias);
      q.pro = o.pro; q.pstats = (const stat_t*)B(o.pstats); q.pgroups = o.pgroups;
      q.pgamma = W(o.pgamma); q.pbeta = W(o.pbeta);
      if (o.pro & PRO_TEMB) {
        q.temb = (const float*)B(P->time_table) + o.temb_col;
        if (row_dev) { q.d_row = row_dev; q.temb_rstride = P->sumC; q.temb_bstride = 0; }
        else { q.d_row = nullptr; q.temb_rstride = 0; q.temb_bstride = P->sumC; }
      }
      if (o.fold) {
        q.pro = PRO_NONE;
        q.pgroups = 1;
        q.fold_s1 = (const float*)(P->wbase + o.fold_off);
        q.fold_s2 = q.fold_s1 + o.Cout;
      }
      q.out = B(o.out); q.res = B(o.res);
      q.ostats = (stat_t*)B(o.ostats); q.ogroups = o.ogroups;
      rc = o.tc ? conv_tcgen05(q, st) : conv_simt(q, P->act, st);
      break;
    }
    case OP_FINALIZE: {
      FinalizeP q;
      q.raw = B(o.raw); q.stats = (const stat_t*)B(o.stats); q.groups = o.groups;
      q.gamma = W(o.gamma); q.beta = W(o.beta); q.silu = o.silu;
      q.res = B(o.res); q.out = B(o.out); q.ostats = (stat_t*)B(o.ostats); q.ogroups = o.ogroups;
      q.B = batch; q.HW = o.HW; q.C = o.C;
      rc = gn_finalize(q, P->act, st);
      break;
    }
    case OP_LINATTN:
      rc = linattn_core(B(o.src1), B(o.out), batch, o.heads, o.dh, o.N, P->act, st);
      break;
    case OP_ATTN:
      rc = attn_core(B(o.src1), B(o.out), batch, o.heads, o.dh, o.N, P->act, st);
      break;
    case OP_ATTN_FUSED: {
      LinAttnFusedP q;
      q.x = B(o.src1); q.out = B(o.out); q.pstats = (const stat_t*)B(o.pstats);
      q.wqkv = P->wbase + P->params[o.w].off;
      q.wo = P->wbase + P->params[o.wo].off;
      q.s1 = (const float*)(P->wbase + o.fold_off);
      q.s2 = q.s1 + 384;
      q.bo = W(o.bo); q.go = W(o.gamma); q.beo = W(o.beta);
      q.B = batch; q.N = o.N; q.C = o.C;
      rc = o.softmax ? attn_softmax_fused(q, st) : linattn_fused(q, st);
      break;
    }
    case OP_CLASSADD:
      rc = class_embed_add(B(o.src1), W(P->pidx["class_embed.weight"]), classes_dev, c.num_classes, batch, o.HW, o.C, P->act, st);
      break;
    case OP_MODULATE:
      rc = film_modulate(B(o.src1), B(o.src2), B(o.res), B(o.out), (long)batch * o.HW * o.C, P->act, st);
      break;
    case OP_FINALPROJ: {
      const FinalProjP q = final_proj_params(P, o, out_dev, batch);
      if (tail) rc = launch_final_proj_ddpm(q, tail->x, tail->z, tail->out, tail->coef, tail->step_dev, tail->step, tail->rng, tail->rng_dev, tail->advance, st);
      else rc = final_proj(q, P->act, st);
      break;
    }
  }
  return rc;
}

static int run_forward(dmn_plan* P, const float* x_dev, const int32_t* row_dev, const int64_t* classes_dev, float* out_dev,
                       int batch, cudaStream_t st, std::vector<cudaEvent_t>* evs = nullptr, const TailFuse* tail = nullptr,
                       unsigned long long* stamps = nullptr) {
  const long launches0 = g_launches;
  size_t op_i = 0;
  if (evs) cudaEventRecord((*evs)[0], st);
  if (stamps) stamp_kernel<<<1, 1, 0, st>>>(stamps);
  for (const Op& o : P->ops) {
    const int rc = enqueue_op(P, o, x_dev, row_dev, classes_dev, out_dev, batch, st, tail);
    if (rc) {
      set_error(o.name + ": " + g_err);
      return rc;
    }
    ++op_i;
    if (evs) cudaEventRecord((*evs)[op_i], st);
    if (stamps) stamp_kernel<<<1, 1, 0, st>>>(stamps + op_i);
  }
  if (stamps) stamp_kernel<<<1, 1, 0, st>>>(stamps + op_i + 1);      // two stamps back to back: the cost of a stamp itself
  P->launches_per_forward = (int)(g_launches - launches0);
  return 0;
}

// ---- forward-mode JVP (fp32 SIMT plans) ----
// The tangent of workspace buffer b lives at work + b.off (same layout as the workspace); behind that arena, a scratch of
// batch * jvp_scratch_per_sample floats holds the materialised operand of a tangent convolution whose primal has a
// GroupNorm(+SiLU) prologue (jvp.cu: gn_tangent).
static size_t jvp_scratch_per_sample(const dmn_plan* P) {
  size_t m = 0;
  for (const Op& o : P->ops) {
    if (o.kind == OP_CONV && (o.pro & PRO_GN)) m = std::max(m, (size_t)o.Hin * o.Hin * o.C1);
    if (o.kind == OP_FINALPROJ && o.groups > 0) m = std::max(m, (size_t)o.HW * o.C);
  }
  return m;
}

static size_t jvp_work_bytes(const dmn_plan* P, int batch) {
  return align_up(P->ws_bytes, 256) + (size_t)batch * jvp_scratch_per_sample(P) * sizeof(float);
}

// the tangent of op o (run right after o itself, while o's primal inputs and outputs are live): v = input tangent (NCHW),
// tan_out = output tangent (NCHW)
static int enqueue_tangent_op(dmn_plan* P, const Op& o, const float* v_dev, float* tan_out, char* work, int batch, cudaStream_t st) {
  auto W = [&](int pi) -> const float* { return pi < 0 ? nullptr : (const float*)(P->wbase + P->params[pi].off); };
  auto B = [&](const Buf& b) -> float* { return b.valid() ? (float*)(P->wsbase + b.off) : nullptr; };
  auto T = [&](const Buf& b) -> float* { return b.valid() ? (float*)(work + b.off) : nullptr; };
  float* du = (float*)(work + align_up(P->ws_bytes, 256));
  auto gn_tan = [&](const float* h, const float* dh, const Buf& stats, int groups, int gamma, int beta, int silu, const float* dres,
                    float* out, int HW, int C) {
    GnTangentP g;
    g.h = h; g.dh = dh; g.stats = (const stat_t*)B(stats); g.groups = groups; g.gamma = W(gamma); g.beta = W(beta); g.silu = silu;
    g.dres = dres; g.out = out; g.B = batch; g.HW = HW; g.C = C;
    return gn_tangent(g, st);
  };
  int rc = 0;
  switch (o.kind) {
    case OP_MEMSET:
      break;
    case OP_INIT: {       // class embedding and bias do not depend on x
      InitConvP q;
      q.x = v_dev;
      q.w = W(P->pidx["init_conv.weight"]);
      q.out = T(o.out);
      q.B = batch; q.Cin = P->cfg.channels; q.S = P->cfg.image_size; q.Cout = P->cfg.dim;
      rc = init_conv(q, ACT_F32, st);
      break;
    }
    case OP_CONV: {
      ConvP q;
      q.src1 = T(o.src1); q.src2 = T(o.src2); q.C1 = o.C1; q.C2 = o.C2;
      q.B = batch; q.Hin = q.Win = o.Hin; q.Hout = q.Wout = o.Hout; q.Cout = o.Cout;
      q.mode = o.mode; q.ksize = o.ksize;
      q.w = P->wbase + P->params[o.w].off;
      if (o.pro & PRO_GN) {    // the time-embedding add of the prologue is constant in x
        if ((rc = gn_tan(B(o.src1), T(o.src1), o.pstats, o.pgroups, o.pgamma, o.pbeta, (o.pro & PRO_SILU) ? 1 : 0, nullptr, du,
                         o.Hin * o.Hin, o.C1)))
          return rc;
        q.src1 = du;
      }
      q.out = T(o.out); q.res = T(o.res);
      rc = conv_simt(q, ACT_F32, st);
      break;
    }
    case OP_FINALIZE:
      rc = gn_tan(B(o.raw), T(o.raw), o.stats, o.groups, o.gamma, o.beta, o.silu, T(o.res), T(o.out), o.HW, o.C);
      break;
    case OP_LINATTN:
      rc = linattn_jvp(B(o.src1), T(o.src1), T(o.out), batch, o.heads, o.dh, o.N, st);
      break;
    case OP_ATTN:
      rc = attn_jvp(B(o.src1), T(o.src1), T(o.out), batch, o.heads, o.dh, o.N, st);
      break;
    case OP_FINALPROJ: {
      FinalProjP q = final_proj_params(P, o, tan_out, batch);
      if (o.groups > 0) {
        if ((rc = gn_tan(B(o.src1), T(o.src1), o.stats, o.groups, o.gamma, o.beta, 1, nullptr, du, o.HW, o.C))) return rc;
        q.y = du;
      } else {
        q.y = T(o.src1);
      }
      q.plain = 1; q.stats = nullptr; q.gamma = q.beta = nullptr; q.bias = nullptr;
      rc = final_proj(q, ACT_F32, st);
      break;
    }
    default:
      return fail(DMN_ENOTSUP, "no tangent for this op (FiLM / fused tensor-core ops)");
  }
  return rc;
}

static int run_jvp(dmn_plan* P, const float* x_dev, const float* v_dev, const int32_t* row_dev, const int64_t* classes_dev, float* out_dev,
                   float* tan_out, char* work, int batch, cudaStream_t st) {
  for (const Op& o : P->ops) {
    int rc = enqueue_op(P, o, x_dev, row_dev, classes_dev, out_dev, batch, st, nullptr);
    if (!rc) rc = enqueue_tangent_op(P, o, v_dev, tan_out, work, batch, st);
    if (rc) {
      set_error(o.name + ": " + g_err);
      return rc;
    }
  }
  return 0;
}

static int check_ready(const dmn_plan* p) {
  if (!p) return fail(DMN_EINVAL, "null plan");
  if (!p->wbase || !p->wsbase) return fail(DMN_ESTATE, "plan is not bound to device memory (dmn_plan_bind)");
  for (const auto& q : p->params)
    if (!q.loaded) return fail(DMN_ESTATE, "parameter not loaded: " + q.name);
  if ((p->cfg.with_time_emb || p->cfg.film) && !p->freqs_loaded)
    return fail(DMN_ESTATE, "sinusoid / FiLM frequencies not loaded (dmn_plan_load_freqs)");
  return 0;
}

// Captures enqueue(stream) on a private non-blocking stream (thread-local capture) and instantiates the graph into *out.
// An error enqueue returns is passed through; a failing CUDA call of the capture itself becomes DMN_ECUDA naming `what`.
template <class Enqueue>
static int capture_graph(const char* what, Enqueue&& enqueue, cudaGraphExec_t* out) {
  cudaStream_t cs;
  DMN_CUDA_CHECK(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
  int rc = 0;
  const char* where = "begin capture";
  cudaGraph_t graph = nullptr;
  cudaError_t e = cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal);
  if (e == cudaSuccess) {
    rc = enqueue(cs);
    const cudaError_t e2 = cudaStreamEndCapture(cs, &graph);
    if (!rc && e2 != cudaSuccess) { where = "end capture"; e = e2; }
  }
  cudaStreamDestroy(cs);
  if (!rc && e == cudaSuccess) { where = "instantiate"; e = cudaGraphInstantiate(out, graph, 0); }
  if (graph) cudaGraphDestroy(graph);
  cudaGetLastError();
  if (rc) return rc;
  if (e != cudaSuccess) return fail(DMN_ECUDA, std::string(what) + " (" + where + "): " + cudaGetErrorString(e));
  return 0;
}

}  // namespace dmn

extern "C" {

const char* dmn_last_error(void) { return g_err.c_str(); }
int dmn_abi_version(void) { return DMN_ABI_VERSION; }

int dmn_plan_create(const dmn_unet_cfg* cfg, dmn_plan** out) {
  if (!cfg || !out) return fail(DMN_EINVAL, "null argument");
  DMN_REQUIRE(cfg->n_mults >= 1 && cfg->n_mults <= 8, "n_mults out of range");
  DMN_REQUIRE(cfg->dim >= 8 && cfg->dim % 8 == 0, "dim must be a multiple of 8");
  DMN_REQUIRE(cfg->groups >= 1 && cfg->dim % cfg->groups == 0 && (cfg->dim / cfg->groups) % 4 == 0,
              "resnet_block_groups must divide dim with at least 4 channels per group");
  DMN_REQUIRE(cfg->channels >= 1 && cfg->channels <= 16 && cfg->out_dim >= 1 && cfg->out_dim <= 8, "channels / out_dim out of range");
  DMN_REQUIRE(cfg->image_size >= 4 && cfg->max_batch >= 1, "image_size / max_batch out of range");
  DMN_REQUIRE(cfg->act_dtype == DMN_ACT_F32 || cfg->act_dtype == DMN_ACT_BF16, "act_dtype");
  DMN_REQUIRE(cfg->conv_engine == DMN_CONV_SIMT || (cfg->conv_engine == DMN_CONV_TCGEN05 && cfg->act_dtype == DMN_ACT_BF16),
              "tcgen05 engine requires bf16 activations");
  DMN_REQUIRE(cfg->with_time_emb == 0 || cfg->with_time_emb == 1, "with_time_emb must be 0 or 1");
  DMN_REQUIRE(cfg->film == 0 || cfg->film == 1, "film must be 0 or 1");
  DMN_REQUIRE(cfg->plain_tail == 0 || cfg->plain_tail == 1, "plain_tail must be 0 or 1");
  for (int i = 0; i < cfg->n_mults; ++i) DMN_REQUIRE(cfg->dim_mults[i] >= 1, "dim_mults must be positive");
  std::unique_ptr<dmn_plan> p(new dmn_plan());
  p->cfg = *cfg;
  if (p->cfg.max_time_rows < p->cfg.max_batch) p->cfg.max_time_rows = p->cfg.max_batch;
  p->act = cfg->act_dtype;
  p->engine = cfg->conv_engine;
  p->esz = cfg->act_dtype == DMN_ACT_F32 ? 4 : 2;
  Builder b(*p);
  int rc = b.build();
  if (rc) return rc;
  *out = p.release();
  return 0;
}

void dmn_plan_destroy(dmn_plan* p) { delete p; }
size_t dmn_plan_weights_bytes(const dmn_plan* p) { return p ? p->weights_bytes : 0; }
size_t dmn_plan_workspace_bytes(const dmn_plan* p) { return p ? p->ws_bytes : 0; }

int dmn_plan_bind(dmn_plan* p, void* weights_dev, size_t weights_bytes, void* workspace_dev, size_t workspace_bytes) {
  if (!p) return fail(DMN_EINVAL, "null plan");
  DMN_REQUIRE(weights_dev && workspace_dev, "null device pointer");
  DMN_REQUIRE(weights_bytes >= p->weights_bytes && workspace_bytes >= p->ws_bytes, "buffers smaller than dmn_plan_*_bytes()");
  DMN_REQUIRE(((uintptr_t)weights_dev % 256) == 0 && ((uintptr_t)workspace_dev % 256) == 0, "device buffers must be 256-byte aligned");
  p->wbase = (char*)weights_dev;
  p->wsbase = (char*)workspace_dev;
  p->drop_graphs();
  return 0;
}

int dmn_plan_num_params(const dmn_plan* p) { return p ? (int)p->params.size() : 0; }
const char* dmn_plan_param_name(const dmn_plan* p, int i) {
  if (!p || i < 0 || i >= (int)p->params.size()) return nullptr;
  return p->params[i].name.c_str();
}
int dmn_plan_param_shape(const dmn_plan* p, int i, int64_t shape_out[4]) {
  if (!p || i < 0 || i >= (int)p->params.size()) return fail(DMN_EINVAL, "bad parameter index");
  const auto& s = p->params[i].shape;
  for (size_t k = 0; k < s.size() && k < 4; ++k) shape_out[k] = s[k];
  return (int)s.size();
}

int dmn_plan_load_param(dmn_plan* p, const char* name, const float* host, int64_t numel, void* stream) {
  if (!p || !name || !host) return fail(DMN_EINVAL, "null argument");
  if (!p->wbase) return fail(DMN_ESTATE, "bind the plan before loading parameters");
  auto it = p->pidx.find(name);
  if (it == p->pidx.end()) return fail(DMN_EINVAL, std::string("unknown parameter: ") + name);
  Param& q = p->params[it->second];
  if (numel != q.numel()) return fail(DMN_EINVAL, std::string("size mismatch for ") + name);
  cudaStream_t st = (cudaStream_t)stream;
  const bool rb = p->act == DMN_ACT_BF16;
  std::vector<float> tmp;
  switch (q.kind) {
    case PK_RAW:
      DMN_CUDA_CHECK(cudaMemcpyAsync(p->wbase + q.off, host, numel * sizeof(float), cudaMemcpyHostToDevice, st));
      break;
    case PK_INIT: {
      const int dim = (int)q.shape[0], ch = (int)q.shape[1];
      tmp.resize(numel);
      init_conv_pack_weights(ch, dim, host, tmp.data());
      DMN_CUDA_CHECK(cudaMemcpyAsync(p->wbase + q.off, tmp.data(), numel * sizeof(float), cudaMemcpyHostToDevice, st));
      if (q.has_tc) {
        std::vector<char> img(init_conv_tcgen05_weight_bytes(dim));
        init_conv_tcgen05_pack_weights(ch, dim, host, img.data());
        DMN_CUDA_CHECK(cudaMemcpyAsync(p->wbase + q.off2, img.data(), img.size(), cudaMemcpyHostToDevice, st));
        DMN_CUDA_CHECK(cudaStreamSynchronize(st));
      }
      break;
    }
    case PK_LIN_T: {
      const int no = (int)q.shape[0], ni = (int)q.shape[1];
      tmp.resize(numel);
      for (int o = 0; o < no; ++o)
        for (int i = 0; i < ni; ++i) tmp[(long)i * no + o] = host[(long)o * ni + i];
      DMN_CUDA_CHECK(cudaMemcpyAsync(p->wbase + q.off, tmp.data(), numel * sizeof(float), cudaMemcpyHostToDevice, st));
      break;
    }
    case PK_BLOCK_MLP_W: {
      const int co = (int)q.shape[0], td = (int)q.shape[1];
      tmp.resize(numel);
      for (int o = 0; o < co; ++o)
        for (int i = 0; i < td; ++i) tmp[(long)i * co + o] = host[(long)o * td + i];
      // strided destination: row i of [4dim][sumC], columns [col, col+co)
      DMN_CUDA_CHECK(cudaMemcpy2DAsync(p->wbase + p->off_wct + (size_t)q.col * sizeof(float), (size_t)p->sumC * sizeof(float),
                                       tmp.data(), (size_t)co * sizeof(float), (size_t)co * sizeof(float), td,
                                       cudaMemcpyHostToDevice, st));
      break;
    }
    case PK_BLOCK_MLP_B:
      DMN_CUDA_CHECK(cudaMemcpyAsync(p->wbase + p->off_bc + (size_t)q.col * sizeof(float), host, numel * sizeof(float),
                                     cudaMemcpyHostToDevice, st));
      break;
    case PK_PLAIN_BF16: {
      if (q.fold_op < 0) {       // folded weights are packed below, once gamma / beta are known too
        std::vector<bf16> img((size_t)numel);
        for (int64_t i = 0; i < numel; ++i) img[i] = __float2bfloat16_rn(host[i]);
        DMN_CUDA_CHECK(cudaMemcpyAsync(p->wbase + q.off, img.data(), img.size() * 2, cudaMemcpyHostToDevice, st));
        DMN_CUDA_CHECK(cudaStreamSynchronize(st));
      }
      break;
    }
    case PK_CONV: {
      if (q.has_simt) {
        tmp.resize(numel);
        conv_simt_pack_weights(q.mode, q.ksize, q.cin, q.cout, host, tmp.data(), rb);
        DMN_CUDA_CHECK(cudaMemcpyAsync(p->wbase + q.off, tmp.data(), numel * sizeof(float), cudaMemcpyHostToDevice, st));
      }
      if (q.has_tc && q.fold_op < 0) {
        const size_t nb = conv_tcgen05_weight_bytes(q.mode, q.ksize, q.cin, q.cout);
        std::vector<char> img(nb);
        conv_tcgen05_pack_weights(q.mode, q.ksize, q.cin, q.cout, host, img.data());
        DMN_CUDA_CHECK(cudaMemcpyAsync(p->wbase + q.off2, img.data(), nb, cudaMemcpyHostToDevice, st));
        DMN_CUDA_CHECK(cudaStreamSynchronize(st));
      }
      break;
    }
  }
  DMN_CUDA_CHECK(cudaStreamSynchronize(st));   // staging buffers are stack-scoped
  q.loaded = true;
  if (q.keep_host) {
    q.host.assign(host, host + numel);
    // folded to_qkv: pack once weight, gamma and beta are all here (any arrival order; re-packed on every reload)
    const Op& o = p->ops[q.fold_op];
    const Param &pw = p->params[o.w], &pg = p->params[o.fold_gamma], &pb = p->params[o.fold_beta];
    if (!pw.host.empty() && !pg.host.empty() && !pb.host.empty()) {
      const int cin = pw.cin, cout = pw.cout;
      std::vector<float> wf((size_t)cout * cin), s12((size_t)2 * cout);
      for (int n = 0; n < cout; ++n) {
        double s1 = 0.0, s2 = 0.0;
        for (int c = 0; c < cin; ++c) {
          const float wg = pw.host[(size_t)n * cin + c] * pg.host[c];
          wf[(size_t)n * cin + c] = wg;
          s1 += (double)__bfloat162float(__float2bfloat16_rn(wg));     // the value the tensor core multiplies with
          s2 += (double)pw.host[(size_t)n * cin + c] * (double)pb.host[c];
        }
        s12[n] = (float)s1;
        s12[cout + n] = (float)s2;
      }
      if (pw.kind == PK_PLAIN_BF16) {        // fused attention block: row-major bf16 [cout][cin]
        std::vector<bf16> img(wf.size());
        for (size_t i = 0; i < wf.size(); ++i) img[i] = __float2bfloat16_rn(wf[i]);
        DMN_CUDA_CHECK(cudaMemcpyAsync(p->wbase + pw.off, img.data(), img.size() * 2, cudaMemcpyHostToDevice, st));
        DMN_CUDA_CHECK(cudaMemcpyAsync(p->wbase + o.fold_off, s12.data(), s12.size() * sizeof(float), cudaMemcpyHostToDevice, st));
        DMN_CUDA_CHECK(cudaStreamSynchronize(st));
      } else {
        std::vector<char> img(conv_tcgen05_weight_bytes(pw.mode, pw.ksize, cin, cout));
        conv_tcgen05_pack_weights(pw.mode, pw.ksize, cin, cout, wf.data(), img.data());
        DMN_CUDA_CHECK(cudaMemcpyAsync(p->wbase + pw.off2, img.data(), img.size(), cudaMemcpyHostToDevice, st));
        DMN_CUDA_CHECK(cudaMemcpyAsync(p->wbase + o.fold_off, s12.data(), s12.size() * sizeof(float), cudaMemcpyHostToDevice, st));
        DMN_CUDA_CHECK(cudaStreamSynchronize(st));
      }
    }
  }
  return 0;
}

int dmn_plan_load_freqs(dmn_plan* p, const float* host_freqs, int n, void* stream) {
  if (!p || !host_freqs) return fail(DMN_EINVAL, "null argument");
  if (!p->wbase) return fail(DMN_ESTATE, "bind the plan before loading parameters");
  if (p->cfg.film) {
    // one frequency per table column (every FiLM layer's [exponents | exponents], parts/film.py:20-24); the sin / cos half mask is built here
    DMN_REQUIRE(n == p->sumC, "expected one frequency per FiLM table column (dmn_plan_film_layout)");
    std::vector<float> is_cos;
    for (int ch : p->film_channels)
      for (int k = 0; k < ch; ++k) is_cos.push_back(k >= ch / 2 ? 1.f : 0.f);
    DMN_CUDA_CHECK(cudaMemcpyAsync(p->wbase + p->off_freqs + (size_t)n * sizeof(float), is_cos.data(), n * sizeof(float),
                                   cudaMemcpyHostToDevice, (cudaStream_t)stream));
  } else {
    DMN_REQUIRE(n == p->cfg.dim / 2, "expected dim/2 frequencies");
  }
  DMN_CUDA_CHECK(cudaMemcpyAsync(p->wbase + p->off_freqs, host_freqs, n * sizeof(float), cudaMemcpyHostToDevice, (cudaStream_t)stream));
  DMN_CUDA_CHECK(cudaStreamSynchronize((cudaStream_t)stream));
  p->freqs_loaded = true;
  return 0;
}

int dmn_plan_ready(const dmn_plan* p) { return check_ready(p) == 0 ? 1 : 0; }

int dmn_plan_film_layout(const dmn_plan* p, int32_t* channels_out, int cap) {
  if (!p) return 0;
  const int n = (int)p->film_channels.size();
  for (int i = 0; i < n && i < cap && channels_out; ++i) channels_out[i] = p->film_channels[i];
  return n;
}

int dmn_time_table(dmn_plan* p, const float* times_dev, int row0, int rows, void* stream) {
  // rows_linear_kernel puts the rows on grid.y; refuse a count it cannot launch before anything is enqueued
  DMN_REQUIRE(rows <= 65535, "dmn_time_table takes at most 65535 rows per call");
  int rc = check_ready(p);
  if (rc) return rc;
  DMN_REQUIRE(times_dev && row0 >= 0 && rows > 0 && row0 + rows <= p->cfg.max_time_rows, "time table rows out of range");
  if (p->cfg.film) {
    const float* fr = (const float*)(p->wbase + p->off_freqs);
    return film_pe_table(times_dev, fr, fr + p->sumC, (float*)(p->wsbase + p->time_table.off) + (size_t)row0 * p->sumC, rows, p->sumC,
                         (cudaStream_t)stream);
  }
  if (!p->cfg.with_time_emb) return 0;     // nothing depends on time (unet.py:68-69)
  const int dim = p->cfg.dim;
  TimeP t;
  t.times = times_dev;
  t.freqs = (const float*)(p->wbase + p->off_freqs);
  t.w1t = (const float*)(p->wbase + p->params[p->pidx["time_mlp.1.weight"]].off);
  t.b1 = (const float*)(p->wbase + p->params[p->pidx["time_mlp.1.bias"]].off);
  t.w3t = (const float*)(p->wbase + p->params[p->pidx["time_mlp.3.weight"]].off);
  t.b3 = (const float*)(p->wbase + p->params[p->pidx["time_mlp.3.bias"]].off);
  t.wct = (const float*)(p->wbase + p->off_wct);
  t.bc = (const float*)(p->wbase + p->off_bc);
  t.tmp = (float*)(p->wsbase + p->time_tmp.off) + (size_t)row0 * 8 * dim;
  t.table = (float*)(p->wsbase + p->time_table.off) + (size_t)row0 * p->sumC;
  t.rows = rows; t.dim = dim; t.sumC = p->sumC;
  return time_table(t, (cudaStream_t)stream);
}

int dmn_plan_time_table_info(const dmn_plan* p, size_t* ws_offset, int32_t* sum_c, int32_t* max_rows) {
  if (!p) return fail(DMN_EINVAL, "null plan");
  DMN_REQUIRE(p->time_table.valid(), "plan has neither a time embedding nor FiLM: no time table");
  if (ws_offset) *ws_offset = p->time_table.off;
  if (sum_c) *sum_c = p->sumC;
  if (max_rows) *max_rows = p->cfg.max_time_rows;
  return 0;
}

int dmn_plan_param_time_col(const dmn_plan* p, int i) {
  if (!p || i < 0 || i >= (int)p->params.size()) return -1;
  const Param& q = p->params[i];
  return (q.kind == PK_BLOCK_MLP_W || q.kind == PK_BLOCK_MLP_B) ? q.col : -1;
}

int dmn_plan_film_col(const dmn_plan* p, int layer) {
  if (!p || layer < 0 || layer >= (int)p->film_cols.size()) return -1;
  return p->film_cols[layer];
}

int dmn_unet_forward(dmn_plan* p, const float* x_dev, const int32_t* row_dev, const int64_t* classes_dev, float* out_dev,
                     int batch, void* stream) {
  int rc = check_ready(p);
  if (rc) return rc;
  DMN_REQUIRE(x_dev && out_dev, "null tensor");
  DMN_REQUIRE(batch >= 1 && batch <= p->cfg.max_batch, "batch exceeds the plan's max_batch");
  return run_forward(p, x_dev, row_dev, classes_dev, out_dev, batch, (cudaStream_t)stream);
}

size_t dmn_unet_jvp_work_bytes(const dmn_plan* p, int batch) {
  if (!p || batch < 1) return 0;
  return jvp_work_bytes(p, batch);
}

int dmn_unet_jvp(dmn_plan* p, const float* x_dev, const float* v_dev, const int32_t* row_dev, const int64_t* classes_dev, float* out_dev,
                 float* out_tangent_dev, void* work_dev, size_t work_bytes, int batch, void* stream) {
  if (!p) return fail(DMN_EINVAL, "null plan");
  if (p->act != DMN_ACT_F32 || p->engine != DMN_CONV_SIMT)
    return fail(DMN_ENOTSUP, "dmn_unet_jvp: the JVP is built for fp32 plans on the SIMT engine only (bf16 / tcgen05 have no tangent kernels)");
  if (p->cfg.film) return fail(DMN_ENOTSUP, "dmn_unet_jvp: FiLM plans (WaveGradUNet) have no tangent program");
  DMN_REQUIRE(x_dev && v_dev && out_dev && out_tangent_dev && work_dev, "null tensor");
  DMN_REQUIRE(batch >= 1 && batch <= p->cfg.max_batch, "batch exceeds the plan's max_batch");
  DMN_REQUIRE(((uintptr_t)work_dev % 256) == 0, "work buffer must be 256-byte aligned");
  int rc = check_ready(p);
  if (rc) return rc;
  DMN_REQUIRE(work_bytes >= jvp_work_bytes(p, batch), "work buffer smaller than dmn_unet_jvp_work_bytes()");
  return run_jvp(p, x_dev, v_dev, row_dev, classes_dev, out_dev, out_tangent_dev, (char*)work_dev, batch, (cudaStream_t)stream);
}

int dmn_plan_launches_per_forward(const dmn_plan* p) { return p ? p->launches_per_forward : 0; }

int dmn_plan_num_ops(const dmn_plan* p) { return p ? (int)p->ops.size() : 0; }

int dmn_plan_op_info(const dmn_plan* p, int i, char* name_out, int name_cap, int32_t* kind, int32_t* engine,
                     double* flops_per_sample, double* bytes_per_sample) {
  if (!p || i < 0 || i >= (int)p->ops.size()) return fail(DMN_EINVAL, "bad op index");
  const Op& o = p->ops[i];
  const dmn_unet_cfg& c = p->cfg;
  const double esz = (double)p->esz;
  double fl = 0, by = 0;
  switch (o.kind) {
    case OP_MEMSET: by = (double)p->stats_bytes / c.max_batch; break;
    case OP_INIT:
      fl = 2.0 * c.image_size * c.image_size * 49.0 * c.channels * c.dim;
      by = 4.0 * c.image_size * c.image_size * c.channels + esz * c.image_size * c.image_size * c.dim;
      break;
    case OP_CONV: {
      const double cin = o.C1 + o.C2;
      const double taps = o.mode == CONV_SAME ? o.ksize * o.ksize : 16.0;
      const double mpix = o.mode == CONV_UP ? (double)o.Hin * o.Hin : (double)o.Hout * o.Hout;   // MACs counted on the strided side
      fl = 2.0 * mpix * taps * cin * o.Cout;
      by = esz * ((double)o.Hin * o.Hin * cin + (double)o.Hout * o.Hout * o.Cout * (o.res.valid() ? 2.0 : 1.0)) + 2.0 * taps * cin * o.Cout / c.max_batch;
      break;
    }
    case OP_FINALIZE: by = esz * (double)o.HW * o.C * 3.0; break;
    case OP_MODULATE: by = esz * (double)o.HW * o.C * 4.0; break;
    case OP_CLASSADD: by = esz * (double)o.HW * o.C * 2.0; break;
    case OP_LINATTN: fl = 2.0 * 2.0 * o.heads * o.dh * o.dh * o.N; by = esz * (double)o.N * o.heads * o.dh * 4.0; break;
    case OP_ATTN: fl = 2.0 * 2.0 * o.heads * o.dh * (double)o.N * o.N; by = esz * (double)o.N * o.heads * o.dh * 4.0; break;
    case OP_FINALPROJ: fl = 2.0 * o.HW * o.C * o.Cout; by = esz * (double)o.HW * o.C + 4.0 * o.HW * o.Cout; break;
    case OP_ATTN_FUSED:      // to_qkv + both contractions + to_out; x read once, result written once
      fl = 2.0 * o.N * (384.0 * o.C + (o.softmax ? 2.0 * 128.0 * o.N : 2.0 * 128.0 * 32.0) + 128.0 * o.C);
      by = esz * (double)o.N * o.C * 2.0;
      break;
  }
  if (name_out && name_cap > 0) {
    strncpy(name_out, o.name.c_str(), (size_t)name_cap - 1);
    name_out[name_cap - 1] = 0;
  }
  if (kind) *kind = o.kind;
  // OP_ATTN in bf16 above 64 tokens runs attn_flash_kernel (tcgen05)
  const bool flash = o.kind == OP_ATTN && p->act == ACT_BF16 && o.N > 64;
  if (engine) *engine = ((o.kind == OP_CONV && o.tc) || (o.kind == OP_INIT && p->init_tc) || o.kind == OP_ATTN_FUSED || flash) ? 1 : 0;
  if (flops_per_sample) *flops_per_sample = fl;
  if (bytes_per_sample) *bytes_per_sample = by;
  return 0;
}

int dmn_plan_profile_forward(dmn_plan* p, const float* x_dev, const int32_t* row_dev, const int64_t* classes_dev,
                             float* out_dev, int batch, void* stream, float* ms_out, int max_ops) {
  int rc = check_ready(p);
  if (rc) return rc;
  DMN_REQUIRE(x_dev && out_dev && ms_out, "null tensor");
  DMN_REQUIRE(batch >= 1 && batch <= p->cfg.max_batch, "batch exceeds the plan's max_batch");
  DMN_REQUIRE(max_ops >= (int)p->ops.size(), "ms_out too small (dmn_plan_num_ops)");
  std::vector<cudaEvent_t> evs(p->ops.size() + 1);
  for (auto& e : evs) DMN_CUDA_CHECK(cudaEventCreate(&e));
  rc = run_forward(p, x_dev, row_dev, classes_dev, out_dev, batch, (cudaStream_t)stream, &evs);
  if (!rc) {
    cudaError_t e = cudaStreamSynchronize((cudaStream_t)stream);
    if (e != cudaSuccess) rc = fail(DMN_ECUDA, std::string("profile_forward: ") + cudaGetErrorString(e));
  }
  if (!rc)
    for (size_t i = 0; i < p->ops.size(); ++i) cudaEventElapsedTime(&ms_out[i], evs[i], evs[i + 1]);
  for (auto& e : evs) cudaEventDestroy(e);
  return rc;
}

/* Same measurement inside ONE CUDA graph: the forward program is stream-captured with an event-record node between
 * consecutive launches, the graph is replayed (once warm, once timed) and the per-launch times are the event differences.
 * Unlike plain stream launches the kernels run back to back as they do in the sampling loop (no exposed launch latency). */
int dmn_plan_profile_forward_graph(dmn_plan* p, const float* x_dev, const int32_t* row_dev, const int64_t* classes_dev,
                                   float* out_dev, int batch, void* stream, float* ms_out, int max_ops) {
  int rc = check_ready(p);
  if (rc) return rc;
  DMN_REQUIRE(x_dev && out_dev && ms_out, "null tensor");
  DMN_REQUIRE(batch >= 1 && batch <= p->cfg.max_batch, "batch exceeds the plan's max_batch");
  DMN_REQUIRE(max_ops >= (int)p->ops.size(), "ms_out too small (dmn_plan_num_ops)");
  const size_t n = p->ops.size();
  // CUDA events recorded by graph nodes cannot be timed (cudaEventElapsedTime: invalid argument), so the stamps are %globaltimer
  // reads of one-thread kernels between the launches; the cost of a stamp (two of them back to back at the end) is subtracted.
  // Measurement aid only: the one other place (besides the GEMM self-test) where the library allocates device memory itself.
  unsigned long long* stamps = nullptr;
  DMN_CUDA_CHECK(cudaMalloc(&stamps, (n + 2) * sizeof(unsigned long long)));
  cudaGraphExec_t exec = nullptr;
  rc = capture_graph("profile_forward_graph", [&](cudaStream_t cs) {
    return run_forward(p, x_dev, row_dev, classes_dev, out_dev, batch, cs, nullptr, nullptr, stamps);
  }, &exec);
  std::vector<unsigned long long> host(n + 2);
  const char* where = "launch";
  cudaError_t e = cudaSuccess;
  if (!rc) {
    cudaStream_t st = (cudaStream_t)stream;
    e = cudaGraphLaunch(exec, st);
    if (e == cudaSuccess) e = cudaGraphLaunch(exec, st);
    if (e == cudaSuccess) { where = "synchronize"; e = cudaStreamSynchronize(st); }
    if (e == cudaSuccess) { where = "copy"; e = cudaMemcpy(host.data(), stamps, (n + 2) * sizeof(unsigned long long), cudaMemcpyDeviceToHost); }
    if (e == cudaSuccess) {
      const double stamp_ns = (double)(host[n + 1] - host[n]);
      for (size_t i = 0; i < n; ++i) {
        double ns = (double)(host[i + 1] - host[i]) - stamp_ns;
        ms_out[i] = (float)((ns > 0 ? ns : 0) * 1e-6);
      }
    }
  }
  if (exec) cudaGraphExecDestroy(exec);
  cudaFree(stamps);
  if (!rc && e != cudaSuccess) rc = fail(DMN_ECUDA, std::string("profile_forward_graph (") + where + "): " + cudaGetErrorString(e));
  cudaGetLastError();
  return rc;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------
// loop driver
// ---------------------------------------------------------------------------------------------------------
// Slack of the loop scratch, in floats: the sizes the loop has always required, from which every offset below derives.
//  kLoopSlack: the tail behind x_mean is 2*batch + kLoopSlack floats; the Langevin norms use 2*batch + 2 of them.
//  kLoopGuidedSlack: with guidance the layout ends 2*batch + kLoopGuidedSlack floats behind its 3*(n_out + n) buffers: the tail
//    rounded up to 4 floats, so x2 and mo2 stay 16-byte aligned for the float4 guidance kernels, then 18 or 20 spare floats.
static constexpr long kLoopSlack = 16, kLoopGuidedSlack = 36;

// views into dmn_loop_desc.scratch_dev; the buffers a descriptor does not use are nullptr
struct LoopWork {
  long chw = 0, n = 0, n_out = 0;        // C*S*S; batch * chw (the state); batch * out_dim*S*S (the model output)
  float* mo = nullptr;                   // [n_out] model output (guidance: the mixed eps)
  float* xmean = nullptr;                // [n] PC: x_mean; BPD: x_t
  float* lscr = nullptr;                 // [2*batch + 2] Langevin norms
  float* x2 = nullptr;                   // guidance: [2n] the doubled batch [x ; x]
  float* mo2 = nullptr;                  // guidance: [2*n_out] its model output
  float* ring = nullptr;                 // DPM-Solver++: [3n] history ring, float4-aligned
};

// floats of scratch the descriptor needs (reads kind, batch and cfg_on); fills w with views into base when given
static size_t loop_work_layout(const dmn_unet_cfg& c, const dmn_loop_desc& d, float* base, LoopWork* w) {
  const auto round4 = [](long v) { return (v + 3) & ~3L; };
  const long chw = (long)c.channels * c.image_size * c.image_size;
  const long n = d.batch * chw;
  const long n_out = (long)d.batch * c.out_dim * c.image_size * c.image_size;
  const long common = d.cfg_on ? 3 * n_out + 3 * n + 2 * d.batch + kLoopGuidedSlack : n_out + n + 2 * d.batch + kLoopSlack;
  const long o_x2 = n_out + n + round4(2 * d.batch + kLoopSlack), o_ring = round4(common);
  const bool dpmpp = d.kind == DMN_LOOP_DPMPP;
  if (w) {
    w->chw = chw; w->n = n; w->n_out = n_out;
    w->mo = base;
    w->xmean = base + n_out;
    w->lscr = base + n_out + n;
    w->x2 = d.cfg_on ? base + o_x2 : nullptr;
    w->mo2 = d.cfg_on ? base + o_x2 + 2 * n : nullptr;
    w->ring = dpmpp ? base + o_ring : nullptr;
  }
  return (size_t)(dpmpp ? o_ring + 3 * n : common);
}

// One loop step.  `ctr` = device step counter (graph mode) or nullptr with host step `s` (injected-noise mode);
// `z0` = this step's injected noise block (draws x n floats) or nullptr for in-kernel Philox with device rng state.
// `ip` (inpainting, never with injected noise): dmn_inpaint_prepare runs first, so everything after it sees the merged state.
static int enqueue_step(dmn_plan* p, const dmn_loop_desc* d, const LoopWork& w, const dmn_inpaint_desc* ip, int32_t* ctr_dev,
                        bool use_ctr, int s, const float* z0, cudaStream_t st) {
  const int32_t* step_dev = use_ctr ? ctr_dev : nullptr;
  const dmn_rng* rng_dev = z0 ? nullptr : reinterpret_cast<const dmn_rng*>(ctr_dev + 4);
  int rc;
  if (ip && (rc = launch_inpaint_prepare(d->state_dev, ip->known_dev, ip->mask_dev, d->state_dev, w.n, ip->prep_coef_dev, step_dev, s,
                                         d->rng, rng_dev, st)))
    return rc;
  if (d->kind == DMN_LOOP_BPD) {
    // bits-per-dimension term of one timestep: x_t ~ q(x_t | x_0), U-Net on x_t, fused KL / decoder-NLL reduction into terms[b][t]
    float* xt = w.xmean;
    if ((rc = launch_bpd_qsample(d->state_dev, z0, xt, w.n, d->coef_dev, step_dev, s, d->rng, rng_dev, st))) return rc;
    if ((rc = run_forward(p, xt, ctr_dev, d->classes_dev, w.mo, d->batch, st))) return rc;
    if ((rc = launch_bpd_term(d->state_dev, xt, w.mo, d->aux_dev, d->batch, w.chw, p->cfg.out_dim == 2 * p->cfg.channels ? 1 : 0,
                              d->n_steps, 0, d->coef_dev, d->coef2_dev, step_dev, s, st)))
      return rc;
    return launch_advance_counter(ctr_dev, st);
  }
  if (d->kind == DMN_LOOP_PC) {
    for (int k = 0; k < d->n_corr; ++k) {
      if ((rc = run_forward(p, d->state_dev, ctr_dev, d->classes_dev, w.mo, d->batch, st))) return rc;
      const float* zk = z0 ? z0 + (long)k * w.n : nullptr;
      if (d->corr_kind == 1)
        rc = launch_affine_noise(d->state_dev, w.mo, zk, d->state_dev, w.xmean, w.n, d->coef2_dev, step_dev, s, k, d->rng, rng_dev, st);
      else
        rc = launch_langevin(d->state_dev, w.mo, zk, d->state_dev, w.xmean, d->batch, w.chw, d->snr, d->coef2_dev, step_dev, s, k,
                             w.lscr, d->rng, rng_dev, st);
      if (rc) return rc;
    }
    if ((rc = run_forward(p, d->state_dev, ctr_dev, d->classes_dev, w.mo, d->batch, st))) return rc;
    const float* zp = z0 ? z0 + (long)d->n_corr * w.n : nullptr;
    if ((rc = launch_affine_noise(d->state_dev, w.mo, zp, d->state_dev, w.xmean, w.n, d->coef_dev, step_dev, s, 7, d->rng, rng_dev, st)))
      return rc;
  } else {
    if (d->cfg_on) {
      // classifier-free guidance: one U-Net evaluation on the doubled batch [x ; x] (labels ; null class), then the mix
      if ((rc = launch_cfg_dup(d->state_dev, w.x2, w.n, st))) return rc;
      if ((rc = run_forward(p, w.x2, ctr_dev, d->classes_dev, w.mo2, 2 * d->batch, st))) return rc;
      // a learned-variance U-Net returns [eps | v] per sample: only eps is guided, v is the conditional branch's
      if ((rc = launch_cfg_combine(w.mo2, w.mo, w.n_out, w.n_out / d->batch, w.chw, d->cfg_scale, st))) return rc;
    } else if (d->kind == DMN_LOOP_DDPM && tail_fusable(p)) {
      // final_conv tail + posterior update (+ step counter unless a trajectory copy still has to see this step's index) in one launch
      TailFuse tf;
      tf.x = d->state_dev; tf.z = z0; tf.out = d->state_dev; tf.coef = d->coef_dev; tf.step_dev = step_dev; tf.step = s;
      tf.rng = d->rng; tf.rng_dev = rng_dev;
      const bool traj = d->traj_dev && d->traj_every > 0;
      tf.advance = traj ? nullptr : ctr_dev;
      if ((rc = run_forward(p, d->state_dev, ctr_dev, d->classes_dev, w.mo, d->batch, st, nullptr, &tf))) return rc;
      if (!traj) return 0;
      if ((rc = launch_traj(d->state_dev, d->traj_dev, w.n, ctr_dev, d->traj_every, d->n_steps, st))) return rc;
      return launch_advance_counter(ctr_dev, st);
    } else if ((rc = run_forward(p, d->state_dev, ctr_dev, d->classes_dev, w.mo, d->batch, st))) {
      return rc;
    }
    if (d->kind == DMN_LOOP_DDPM)
      rc = launch_ddpm(d->state_dev, w.mo, z0, d->state_dev, w.n, d->coef_dev, step_dev, s, d->rng, rng_dev, st);
    else if (d->kind == DMN_LOOP_LEARNED)
      rc = launch_learned(d->state_dev, w.mo, z0, d->state_dev, d->batch, w.chw, d->coef_dev, step_dev, s, d->rng, rng_dev, st);
    else if (d->kind == DMN_LOOP_DDIM)
      rc = launch_ddim(d->state_dev, w.mo, z0, d->state_dev, w.n, d->coef_dev, step_dev, s, d->rng, rng_dev, st);
    else
      rc = launch_dpmpp(d->state_dev, w.mo, w.ring, d->state_dev, d->batch, w.chw, w.n_out / d->batch, d->coef_dev, d->coef2_dev, z0,
                        step_dev, s, d->rng, rng_dev, st);
    if (rc) return rc;
  }
  if (d->traj_dev && d->traj_every > 0)
    if ((rc = launch_traj(d->state_dev, d->traj_dev, w.n, ctr_dev, d->traj_every, d->n_steps, st))) return rc;
  return launch_advance_counter(ctr_dev, st);
}

// the graph bakes in every pointer and scalar below; the RNG seed is NOT baked (it lives in device memory)
static bool same_graph_key(const dmn_loop_desc& a, const dmn_inpaint_desc& ia, const dmn_loop_desc& b, const dmn_inpaint_desc& ib) {
  const bool traj = a.traj_dev || b.traj_dev;   // only the trajectory kernel bakes n_steps in
  return a.kind == b.kind && (!traj || a.n_steps == b.n_steps) && a.batch == b.batch && a.n_corr == b.n_corr && a.snr == b.snr &&
         a.corr_kind == b.corr_kind && a.coef_dev == b.coef_dev && a.coef2_dev == b.coef2_dev && a.classes_dev == b.classes_dev &&
         a.state_dev == b.state_dev && a.scratch_dev == b.scratch_dev && a.traj_dev == b.traj_dev && a.traj_every == b.traj_every &&
         a.cfg_scale == b.cfg_scale && a.cfg_on == b.cfg_on && (a.kind != DMN_LOOP_BPD || (a.aux_dev == b.aux_dev && a.n_steps == b.n_steps)) &&
         ia.known_dev == ib.known_dev && ia.mask_dev == ib.mask_dev && ia.prep_coef_dev == ib.prep_coef_dev;
}

// the loop driver of dmn_sample_loop (ip = nullptr) and dmn_sample_loop_inpaint
static int run_loop(dmn_plan* p, const dmn_loop_desc* d, const dmn_inpaint_desc* ip, void* stream) {
  int rc = check_ready(p);
  if (rc) return rc;
  if (!d) return fail(DMN_EINVAL, "null descriptor");
  const dmn_unet_cfg& c = p->cfg;
  DMN_REQUIRE(d->kind >= DMN_LOOP_DDPM && d->kind <= DMN_LOOP_DPMPP, "unknown loop kind");
  DMN_REQUIRE(d->kind != DMN_LOOP_BPD || (d->aux_dev && d->coef2_dev && !d->cfg_on && !d->traj_dev),
              "BPD loop needs the terms buffer (aux_dev) and the second coefficient table; no guidance / trajectory");
  DMN_REQUIRE(d->batch >= 1 && d->batch <= c.max_batch, "batch exceeds the plan's max_batch");
  DMN_REQUIRE(d->n_steps >= 1 && d->n_steps <= c.max_time_rows, "n_steps exceeds the plan's time table");
  DMN_REQUIRE(d->state_dev && d->scratch_dev && d->coef_dev, "null device pointer in loop descriptor");
  DMN_REQUIRE(d->kind != DMN_LOOP_PC || d->n_corr == 0 || d->coef2_dev, "PC loop needs corrector coefficients");
  DMN_REQUIRE(d->n_corr >= 0 && d->n_corr <= 6, "n_corr out of range (0..6)");
  if (d->kind == DMN_LOOP_LEARNED) DMN_REQUIRE(c.out_dim == 2 * c.channels, "learned-variance loop needs a U-Net with 2*channels outputs");
  else if (d->kind == DMN_LOOP_BPD) DMN_REQUIRE(c.out_dim == c.channels || c.out_dim == 2 * c.channels, "BPD: out_dim must be C or 2C");
  else if (d->kind == DMN_LOOP_DPMPP)
    DMN_REQUIRE(c.out_dim == c.channels || c.out_dim == 2 * c.channels, "DPM-Solver++: out_dim must be C or 2C");
  else DMN_REQUIRE(c.out_dim == c.channels, "U-Net out_dim must equal channels for this sampler");
  LoopWork w;
  const size_t scratch_floats = loop_work_layout(c, *d, d->scratch_dev, &w);
  DMN_REQUIRE(d->state_elems == 0 || d->state_elems == w.n, "state_dev does not hold batch * channels * image_size^2 floats for this plan");
  if (d->cfg_on) {
    DMN_REQUIRE(d->kind != DMN_LOOP_PC, "classifier-free guidance is built for the DDPM / learned / DDIM / DPM-Solver++ loops");
    DMN_REQUIRE(c.num_classes >= 0 && d->classes_dev, "classifier-free guidance needs a class-conditional U-Net and 2*batch labels");
    DMN_REQUIRE(2 * d->batch <= c.max_batch, "classifier-free guidance doubles the batch: plan max_batch too small");
    DMN_REQUIRE(w.n % 4 == 0 && w.n_out % 4 == 0, "guidance kernels need 16-byte multiples");
  }
  DMN_REQUIRE(d->scratch_bytes >= scratch_floats * sizeof(float), "loop scratch smaller than dmn_loop_scratch_bytes()");
  cudaStream_t st = (cudaStream_t)stream;
  int32_t* ctr = (int32_t*)(p->wsbase + p->counters.off);
  if ((rc = launch_set_counter(ctr, 0, d->rng, st))) return rc;

  if (d->noise_dev) {
    // parity mode: injected noise => per-step pointers differ, plain launches with the host step index
    const int draws = (d->kind == DMN_LOOP_PC) ? d->n_corr + 1 : (d->kind == DMN_LOOP_DPMPP && !d->coef2_dev ? 0 : 1);
    for (int s = 0; s < d->n_steps; ++s)
      if ((rc = enqueue_step(p, d, w, ip, ctr, false, s, d->noise_dev + (long)s * draws * w.n, st))) return rc;
  } else if (!d->use_graph) {
    for (int s = 0; s < d->n_steps; ++s)
      if ((rc = enqueue_step(p, d, w, ip, ctr, true, 0, nullptr, st))) return rc;
  } else {
    const dmn_inpaint_desc ip_key = ip ? *ip : dmn_inpaint_desc{};
    cudaGraphExec_t exec = nullptr;
    for (auto& g : p->graphs)
      if (same_graph_key(g.key, g.ip, *d, ip_key)) exec = g.exec;
    if (!exec) {
      if ((rc = capture_graph("sample loop graph", [&](cudaStream_t cs) { return enqueue_step(p, d, w, ip, ctr, true, 0, nullptr, cs); },
                              &exec)))
        return rc;
      if (p->graphs.size() >= 8) {
        cudaGraphExecDestroy(p->graphs.front().exec);
        p->graphs.erase(p->graphs.begin());
      }
      dmn_plan::GraphEntry ge;
      ge.exec = exec;
      ge.key = *d;
      ge.ip = ip_key;
      p->graphs.push_back(ge);
    }
    for (int s = 0; s < d->n_steps; ++s) DMN_CUDA_CHECK(cudaGraphLaunch(exec, st));
  }
  if (d->kind == DMN_LOOP_PC && d->aux_dev)
    DMN_CUDA_CHECK(cudaMemcpyAsync(d->aux_dev, w.xmean, w.n * sizeof(float), cudaMemcpyDeviceToDevice, st));
  return 0;
}

extern "C" {

int dmn_sample_loop(dmn_plan* p, const dmn_loop_desc* d, void* stream) { return run_loop(p, d, nullptr, stream); }

size_t dmn_loop_scratch_bytes(const dmn_plan* p, const dmn_loop_desc* d) {
  if (!p || !d || d->kind < DMN_LOOP_DDPM || d->kind > DMN_LOOP_DPMPP || d->batch < 1) return 0;
  return loop_work_layout(p->cfg, *d, nullptr, nullptr) * sizeof(float);
}

int dmn_sample_loop_inpaint(dmn_plan* p, const dmn_loop_desc* d, const dmn_inpaint_desc* ip, void* stream) {
  if (!d || !ip) return fail(DMN_EINVAL, "null descriptor");
  DMN_REQUIRE(d->kind == DMN_LOOP_DDPM || d->kind == DMN_LOOP_LEARNED || d->kind == DMN_LOOP_DDIM,
              "inpainting is built for the DDPM / learned-variance / DDIM loops");
  DMN_REQUIRE(!d->noise_dev, "inpainting has no injected-noise mode: noise_dev must be NULL");
  DMN_REQUIRE(ip->known_dev && ip->mask_dev && ip->prep_coef_dev, "null device pointer in inpaint descriptor");
  int rc = run_loop(p, d, ip, stream);
  if (rc) return rc;
  // final composite: row n_steps = {1, 0, 1, 0} puts the known pixels back exactly and draws nothing
  LoopWork w;
  loop_work_layout(p->cfg, *d, d->scratch_dev, &w);
  return launch_inpaint_prepare(d->state_dev, ip->known_dev, ip->mask_dev, d->state_dev, w.n, ip->prep_coef_dev, nullptr, d->n_steps,
                                d->rng, nullptr, (cudaStream_t)stream);
}

int dmn_loop_launches_per_step(const dmn_plan* p, const dmn_loop_desc* d) {
  if (!p || !d) return 0;
  const int per_fwd = (int)p->ops.size() - 1;   // kernels only: the statistics memset is not counted
  int n = 0;
  if (d->kind == DMN_LOOP_BPD) return per_fwd + 3;
  if (d->kind == DMN_LOOP_PC) n = (d->n_corr + 1) * per_fwd + d->n_corr * (d->corr_kind == 1 ? 1 : 3) + 1;
  else if (d->kind == DMN_LOOP_DDPM && !d->cfg_on && tail_fusable(p)) {
    // fused tail: the update (and, without trajectory capture, the counter) ride on the last launch of the forward program
    return (d->traj_dev && d->traj_every > 0) ? per_fwd + 2 : per_fwd;
  } else n = per_fwd + 1 + (d->cfg_on ? 2 : 0);   // one update kernel: DDPM (unfused), learned, DDIM, DPM-Solver++
  if (d->traj_dev && d->traj_every > 0) n += 1;
  return n + 1;   // + advance_counter
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------
// probability-flow ODE driver (kernels: ode.cu)
// ---------------------------------------------------------------------------------------------------------
// One RK45 attempt: the input of stage 1, the 6 stage rows of the time table, then per stage the model evaluation and the stage
// kernel, then the controller (accept / reject, next step, WHILE condition).  eval(row, stream) evaluates the model at U-Net input
// w.x32 with time-table row w.rows[row] and writes what the stage kernels read (w.mo: the model output, plus the drift of the
// log-density rows for the likelihood).
template <class Eval>
static int enqueue_ode_attempt(dmn_plan* p, const OdeWork& w, const OdeParams& P, cudaGraphConditionalHandle hnd, int use_cond,
                               cudaStream_t st, Eval& eval) {
  int rc;
  if ((rc = launch_ode_stage(w, P, 0, st))) return rc;
  if ((rc = dmn_time_table(p, w.rec->labels, 0, 6, st))) return rc;
  for (int s = 1; s <= 6; ++s) {
    if ((rc = eval(s - 1, st))) return rc;
    if ((rc = launch_ode_stage(w, P, s, st))) return rc;
  }
  return launch_ode_control(w, P, hnd, use_cond, st);
}

// init phase: y0, f0 = f(t0, y0), select_initial_step (one more evaluation), first attempt's stage rows
template <class Eval>
static int enqueue_ode_init(dmn_plan* p, const float* state, const OdeWork& w, const OdeParams& P, cudaGraphConditionalHandle hnd,
                            int use_cond, cudaStream_t st, Eval& eval) {
  int rc;
  if ((rc = launch_ode_init(w, P, st))) return rc;
  if ((rc = launch_ode_init_elem(w, P, state, 0, st))) return rc;
  for (int k = 0; k < 2; ++k) {
    if ((rc = dmn_time_table(p, w.rec->labels, 0, 6, st))) return rc;
    if ((rc = eval(0, st))) return rc;
    if ((rc = launch_ode_init_elem(w, P, nullptr, k == 0 ? 1 : 3, st))) return rc;
    if ((rc = launch_ode_init_step(w, P, k, hnd, use_cond && k == 1, st))) return rc;
    if (k == 0 && (rc = launch_ode_init_elem(w, P, nullptr, 2, st))) return rc;
  }
  return 0;
}

// the graph bakes in every pointer and scalar of the descriptor
static bool same_ode_inputs(const dmn_ode_desc&, const dmn_ode_desc&) { return true; }
static bool same_ode_inputs(const dmn_ode_likelihood_desc& a, const dmn_ode_likelihood_desc& b) { return a.noise_dev == b.noise_dev; }
template <class Desc>
static bool same_ode_key(const Desc& a, const Desc& b) {
  return a.sde_kind == b.sde_kind && a.N == b.N && a.beta_0 == b.beta_0 && a.beta_1 == b.beta_1 && a.sigma_min == b.sigma_min &&
         a.sigma_max == b.sigma_max && a.t0 == b.t0 && a.t1 == b.t1 && a.rtol == b.rtol && a.atol == b.atol && a.max_nfe == b.max_nfe &&
         a.batch == b.batch && a.classes_dev == b.classes_dev && a.state_dev == b.state_dev && a.work_dev == b.work_dev &&
         a.result_dev == b.result_dev;
}

// init phase on the captured stream, then a WHILE node whose body (one attempt) is captured on a second stream, then the finish
template <class Eval>
static int build_ode_graph(dmn_plan* p, float* state, const OdeWork& w, const OdeParams& P, Eval& eval, cudaGraphExec_t* out) {
  cudaStream_t bs;
  DMN_CUDA_CHECK(cudaStreamCreateWithFlags(&bs, cudaStreamNonBlocking));
  auto enqueue = [&](cudaStream_t cs) -> int {
    cudaStreamCaptureStatus cst;
    cudaGraph_t graph = nullptr;
    const cudaGraphNode_t* deps = nullptr;
    size_t ndeps = 0;
    cudaGraphConditionalHandle hnd = 0;
    DMN_CUDA_CHECK(cudaStreamGetCaptureInfo(cs, &cst, nullptr, &graph, &deps, &ndeps));
    DMN_CUDA_CHECK(cudaGraphConditionalHandleCreate(&hnd, graph, 0, cudaGraphCondAssignDefault));
    int rc = enqueue_ode_init(p, state, w, P, hnd, 1, cs, eval);
    if (rc) return rc;
    DMN_CUDA_CHECK(cudaStreamGetCaptureInfo(cs, &cst, nullptr, &graph, &deps, &ndeps));
    cudaGraphNodeParams np = {};
    np.type = cudaGraphNodeTypeConditional;
    np.conditional.handle = hnd;
    np.conditional.type = cudaGraphCondTypeWhile;
    np.conditional.size = 1;
    cudaGraphNode_t node = nullptr;
    DMN_CUDA_CHECK(cudaGraphAddNode(&node, graph, deps, ndeps, &np));
    DMN_CUDA_CHECK(cudaStreamUpdateCaptureDependencies(cs, &node, 1, cudaStreamSetCaptureDependencies));
    cudaGraph_t body = np.conditional.phGraph_out[0];
    DMN_CUDA_CHECK(cudaStreamBeginCaptureToGraph(bs, body, nullptr, nullptr, 0, cudaStreamCaptureModeThreadLocal));
    rc = enqueue_ode_attempt(p, w, P, hnd, 1, bs, eval);
    const cudaError_t e = cudaStreamEndCapture(bs, &body);
    if (rc) return rc;
    if (e != cudaSuccess) return fail(DMN_ECUDA, std::string("ode graph (body end capture): ") + cudaGetErrorString(e));
    return launch_ode_finish(w, state, cs);
  };
  const int rc = capture_graph("ode graph", enqueue, out);
  cudaStreamDestroy(bs);
  return rc;
}

// plain launches: the init phase, then one attempt at a time with a host read of the status in between
template <class Eval>
static int run_ode_plain(dmn_plan* p, float* state, const OdeWork& w, const OdeParams& P, Eval& eval, cudaStream_t st) {
  int rc;
  if ((rc = enqueue_ode_init(p, state, w, P, 0, 0, st, eval))) return rc;
  dmn_ode_result r;
  for (long it = 0;; ++it) {
    DMN_CUDA_CHECK(cudaMemcpyAsync(&r, w.result, sizeof(r), cudaMemcpyDeviceToHost, st));
    DMN_CUDA_CHECK(cudaStreamSynchronize(st));
    if (r.status != DMN_ODE_RUNNING) break;
    if (it > (long)P.max_nfe) return fail(DMN_ESTATE, "ODE controller did not stop within max_nfe");
    if ((rc = enqueue_ode_attempt(p, w, P, 0, 0, st, eval))) return rc;
  }
  return launch_ode_finish(w, state, st);
}

// descriptor checks and solver constants shared by the sampler and the likelihood (their descriptors share these fields)
template <class Desc>
static int check_ode_desc(const dmn_plan* p, const Desc* d) {
  const dmn_unet_cfg& c = p->cfg;
  DMN_REQUIRE(d->sde_kind == DMN_SDE_VP || d->sde_kind == DMN_SDE_VE, "unknown SDE kind");
  if (d->sde_kind == DMN_SDE_VP) DMN_REQUIRE(d->N >= 1 && std::isfinite(d->beta_0) && std::isfinite(d->beta_1), "VP-SDE needs N >= 1 and finite betas");
  else DMN_REQUIRE(d->sigma_min > 0 && d->sigma_max > 0 && std::isfinite(d->sigma_min) && std::isfinite(d->sigma_max), "VE-SDE needs positive sigmas");
  DMN_REQUIRE(std::isfinite(d->t0) && std::isfinite(d->t1) && d->t0 != d->t1, "t0 and t1 must be finite and different");
  DMN_REQUIRE(std::isfinite(d->rtol) && d->rtol > 0 && std::isfinite(d->atol) && d->atol >= 0, "tolerances: rtol > 0, atol >= 0, finite");
  DMN_REQUIRE(d->max_nfe >= 2, "max_nfe must be >= 2 (the initial step selection evaluates twice)");
  DMN_REQUIRE(d->batch >= 1 && d->batch <= c.max_batch, "batch exceeds the plan's max_batch");
  DMN_REQUIRE(d->state_dev && d->work_dev && d->result_dev, "null device pointer in ODE descriptor");
  DMN_REQUIRE(((uintptr_t)d->work_dev % 256) == 0, "work buffer must be 256-byte aligned");
  return 0;
}

template <class Desc>
static OdeParams ode_params(const Desc* d) {
  OdeParams P;
  P.sde_kind = d->sde_kind; P.N = d->N; P.max_nfe = d->max_nfe;
  P.beta_0 = d->beta_0; P.beta_1 = d->beta_1; P.sigma_min = d->sigma_min; P.sigma_max = d->sigma_max;
  P.t0 = d->t0; P.t1 = d->t1; P.atol = d->atol;
  P.rtol = d->rtol < 100 * DBL_EPSILON ? 100 * DBL_EPSILON : d->rtol;     // scipy validate_tol
  return P;
}

// the cached graph of descriptor d (built with build() on a miss; at most 4 per plan and kind), launched on st
template <class Desc, class Build>
static int launch_ode_graph(std::vector<dmn_plan::OdeGraphEntry<Desc>>& cache, const Desc* d, Build&& build, cudaStream_t st) {
  cudaGraphExec_t exec = nullptr;
  for (auto& g : cache)
    if (same_ode_key(g.key, *d) && same_ode_inputs(g.key, *d)) exec = g.exec;
  if (!exec) {
    int rc = build(&exec);
    if (rc) return rc;
    if (cache.size() >= 4) {
      cudaGraphExecDestroy(cache.front().exec);
      cache.erase(cache.begin());
    }
    dmn_plan::OdeGraphEntry<Desc> ge;
    ge.exec = exec;
    ge.key = *d;
    cache.push_back(ge);
  }
  DMN_CUDA_CHECK(cudaGraphLaunch(exec, st));
  return 0;
}

// likelihood work: the RK45 work of the augmented state, then the Hutchinson noise, the JVP output and the JVP work
static size_t lik_work_layout(const dmn_plan* p, int batch, char* base, OdeWork* w, char** jvp_work) {
  const dmn_unet_cfg& c = p->cfg;
  const long nx = (long)batch * c.channels * c.image_size * c.image_size;
  size_t off = align_up(ode_work_layout(nx + batch, base, w), 256);
  const size_t o_eps = off;  off += align_up((size_t)nx * sizeof(float), 256);
  const size_t o_dmo = off;  off += align_up((size_t)nx * sizeof(float), 256);
  const size_t o_jvp = off;  off += jvp_work_bytes(p, batch);
  if (w) {
    w->nx = nx;
    w->eps = (const float*)(base + o_eps);
    w->dmo = (float*)(base + o_dmo);
    *jvp_work = base + o_jvp;
  }
  return off;
}

extern "C" {

size_t dmn_ode_work_bytes(const dmn_plan* p, int batch) {
  if (!p || batch < 1) return 0;
  const dmn_unet_cfg& c = p->cfg;
  return ode_work_layout((long)batch * c.channels * c.image_size * c.image_size, nullptr, nullptr);
}

int dmn_ode_sample(dmn_plan* p, const dmn_ode_desc* d, void* stream) {
  if (!p) return fail(DMN_EINVAL, "null plan");
  if (!d) return fail(DMN_EINVAL, "null descriptor");
  const dmn_unet_cfg& c = p->cfg;
  int rc = check_ode_desc(p, d);
  if (rc) return rc;
  const long n = (long)d->batch * c.channels * c.image_size * c.image_size;
  DMN_REQUIRE(d->state_elems == n, "state_dev does not hold batch * channels * image_size^2 floats for this plan");
  DMN_REQUIRE(d->work_bytes >= dmn_ode_work_bytes(p, d->batch), "work buffer smaller than dmn_ode_work_bytes()");
  DMN_REQUIRE(c.out_dim == c.channels && !c.film, "the ODE drift needs a U-Net with out_dim == channels (no FiLM)");
  DMN_REQUIRE(c.max_time_rows >= 6, "the plan's time table needs >= 6 rows (one per stage of an attempt)");
  if ((rc = check_ready(p))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const OdeParams P = ode_params(d);
  OdeWork w;
  ode_work_layout(n, (char*)d->work_dev, &w);
  w.result = d->result_dev;
  auto eval = [&](int row, cudaStream_t s) { return run_forward(p, w.x32, w.rows + row, d->classes_dev, w.mo, d->batch, s); };
  if (!d->use_graph) return run_ode_plain(p, d->state_dev, w, P, eval, st);
  return launch_ode_graph(p->ode_graphs, d, [&](cudaGraphExec_t* e) { return build_ode_graph(p, d->state_dev, w, P, eval, e); }, st);
}

size_t dmn_ode_likelihood_work_bytes(const dmn_plan* p, int batch) {
  if (!p || batch < 1) return 0;
  return lik_work_layout(p, batch, nullptr, nullptr, nullptr);
}

int dmn_ode_likelihood(dmn_plan* p, const dmn_ode_likelihood_desc* d, void* stream) {
  if (!p) return fail(DMN_EINVAL, "null plan");
  if (!d) return fail(DMN_EINVAL, "null descriptor");
  const dmn_unet_cfg& c = p->cfg;
  if (p->act != DMN_ACT_F32 || p->engine != DMN_CONV_SIMT)
    return fail(DMN_ENOTSUP, "dmn_ode_likelihood: the U-Net JVP is built for fp32 plans on the SIMT engine only");
  int rc = check_ode_desc(p, d);
  if (rc) return rc;
  DMN_REQUIRE(d->hutchinson == DMN_HUTCH_RADEMACHER || d->hutchinson == DMN_HUTCH_GAUSSIAN, "unknown Hutchinson noise type");
  const long nx = (long)d->batch * c.channels * c.image_size * c.image_size;
  DMN_REQUIRE(d->state_elems == nx + d->batch, "state_dev does not hold batch * (channels * image_size^2 + 1) floats for this plan");
  DMN_REQUIRE(d->noise_dev || nx % 4 == 0, "in-kernel Hutchinson noise needs batch * channels * image_size^2 % 4 == 0");
  DMN_REQUIRE(d->work_bytes >= dmn_ode_likelihood_work_bytes(p, d->batch), "work buffer smaller than dmn_ode_likelihood_work_bytes()");
  DMN_REQUIRE(c.out_dim == c.channels && !c.film, "the ODE drift needs a U-Net with out_dim == channels (no FiLM)");
  DMN_REQUIRE(c.max_time_rows >= 6, "the plan's time table needs >= 6 rows (one per stage of an attempt)");
  if ((rc = check_ready(p))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const OdeParams P = ode_params(d);
  OdeWork w;
  char* jvp_work = nullptr;
  lik_work_layout(p, d->batch, (char*)d->work_dev, &w, &jvp_work);
  w.result = d->result_dev;
  float* eps_buf = const_cast<float*>(w.eps);
  if (d->noise_dev) w.eps = d->noise_dev;
  // one JVP pass in direction eps: the model output for the x rows, then the divergence rows
  auto eval = [&](int row, cudaStream_t s) {
    const int r = run_jvp(p, w.x32, w.eps, w.rows + row, d->classes_dev, w.mo, w.dmo, jvp_work, d->batch, s);
    return r ? r : launch_ode_div(w, P, row, d->batch, s);
  };
  // the Hutchinson draw, once per solve on the stream ahead of the solve (the graph reads it from the work buffer)
  auto draw = [&](cudaStream_t s) -> int {
    if (d->noise_dev) return 0;
    int r = dmn_randn(eps_buf, nx, d->rng, 0, s);
    if (!r && d->hutchinson == DMN_HUTCH_RADEMACHER) r = launch_ode_rademacher(eps_buf, nx, s);
    return r;
  };
  if ((rc = draw(st))) return rc;
  if (!d->use_graph) return run_ode_plain(p, d->state_dev, w, P, eval, st);
  return launch_ode_graph(p->lik_graphs, d, [&](cudaGraphExec_t* e) { return build_ode_graph(p, d->state_dev, w, P, eval, e); }, st);
}

}  // extern "C"
