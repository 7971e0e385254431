// Host-side construction of the layer programs, pack tables and weight-gradient job tables
// (see hn_mlp_program.h).  Pure host code.
#include <string.h>
#include <algorithm>
#include "hn_api_internal.h"
#include "hn_mlp_program.h"

namespace hn {

int validate_desc(const hn_model_desc& d) {
  if (is_static(d)) {
    if (d.xyz_freqs != 10 || d.view_freqs != 4)
      return set_error(-11, "hn_model_desc: the static NeRF kernels are instantiated for xyz / dir freqs 10 / 4 (models/nerf.py defaults)");
    return 0;
  }
  const bool se3 = (d.flags & HN_FLAG_WARP_SE3) != 0;
  const bool warp = (d.flags & HN_FLAG_WARP_TRANSLATION) != 0 || se3;
  if (se3 && (d.flags & HN_FLAG_WARP_TRANSLATION))
    return set_error(-10, "hn_model_desc: the warp field is either a TranslationField or an SE3Field");
  const bool bendy = (d.flags & HN_FLAG_SLICE_BENDY) != 0, axis = (d.flags & HN_FLAG_SLICE_AXIS) != 0;
  const bool cond = (d.flags & (HN_FLAG_ALPHA_COND | HN_FLAG_RGB_COND)) != 0;
  if (warp && (bendy == axis))
    return set_error(-10, "hn_model_desc: a warped model needs exactly one of bendy_sheet / axis_aligned_plane slicing "
                          "(slice 'none' with warp is broken in the reference, models.py:269-270)");
  if (!warp && (bendy || axis))
    return set_error(-10, "hn_model_desc: without warp map_points returns the raw points (models.py:568-569): pass no slicing flag");
  if (d.xyz_freqs != 10 || d.view_freqs < 0 || d.view_freqs > kMaxViewFreqs)
    return set_error(-11, "hn_model_desc: kernels are instantiated for xyz freqs 10 and view freqs <= 6");
  if (se3 && axis) {
    if (d.glo_dim != 8 || d.hyper_dim != 8 || d.hyper_freqs != 6 || d.warp_freqs != kSe3Freqs)
      return set_error(-11, "hn_model_desc: the SE3 warp is instantiated for axis_aligned_plane slicing with G = hyper_dim = 8, "
                            "hyper freqs 6 and posenc(points, 0, 8) (warp_freqs = 8; warping.py:150-151)");
  } else if (se3) {
    if (d.glo_dim != 8 || d.hyper_dim != 2 || d.hyper_freqs != 6 || d.warp_freqs != kSe3Freqs || d.sheet_freqs != 7)
      return set_error(-11, "hn_model_desc: the SE3 warp with bendy_sheet slicing is instantiated for G = 8, hyper_dim 2, hyper "
                            "freqs 6, sheet freqs 7 and posenc(points, 0, 8) (warp_freqs = 8); add an instantiation in hn_mlp.cu "
                            "for other shapes");
  } else if (warp) {
    if (d.glo_dim != 8 || d.hyper_freqs != 6 || d.warp_freqs != 10 || d.sheet_freqs != 7)
      return set_error(-11, "hn_model_desc: kernels are instantiated for G=8, hyper freqs 6 (warp 10, sheet 7); add an "
                            "instantiation in hn_mlp.cu for other shapes");
    if (d.hyper_dim != 2 && d.hyper_dim != 4 && d.hyper_dim != 8)
      return set_error(-11, "hn_model_desc: kernels are instantiated for hyper_dim 2, 4 and 8");
    if (axis && d.hyper_dim != d.glo_dim)
      return set_error(-11, "hn_model_desc: axis_aligned_plane needs hyper_dim == glo_dim (the hyper point is the GLO vector, "
                            "models.py:533-534)");
  } else if (cond && d.glo_dim != 8) {
    return set_error(-11, "hn_model_desc: kernels are instantiated for G=8");
  }
  if ((warp || cond) && d.num_embeddings <= 0) return set_error(-12, "hn_model_desc: num_embeddings must be positive");
  return 0;
}

namespace {

struct Builder {
  Program* p;
  LogicalOps* lg;
  uint32_t w16 = 0;  // running weight offset (16-byte units)
  int ones_col = -1; // folded-bias forward programs: INB column of the ones chunk pair (every op gets a bias K step)
  int lg_chunks = 0, lg_total = 0;   // chunk cursor inside / chunk count of the logical matrix being emitted
  void begin_layer(uint8_t epi, int n_out, int bias_off, uint16_t save_chunk, uint16_t mask_chunk, uint16_t gate_word = kNone) {
    Layer& L = p->layers[p->nlayers++];
    L.op0 = (uint8_t)p->nops; L.nops = 0; L.epi = epi; L.pad = 0;
    L.n_out = (uint16_t)n_out; L.bias_off = (uint16_t)bias_off; L.save_chunk = save_chunk; L.mask_chunk = mask_chunk;
    L.gate_word = gate_word; L.pad2 = 0;
  }
  void emit(int n, int k, Src s, int a_col, int tmem_col, int acc_init, int kc0, int kc_total) {
    MmaOp& o = p->ops[p->nops++];
    o.kc0 = (uint16_t)kc0; o.kc_total = (uint16_t)kc_total;
    o.w_off16 = w16; o.n = (uint16_t)n; o.k = (uint16_t)k; o.a_chunk = (uint16_t)(a_col / 8);
    o.tmem_col = (uint16_t)tmem_col; o.src = s; o.acc_init = (uint8_t)acc_init; o.pad = 0;
    int cps = (kStageBytes / (n * 16)) & ~1;
    if (cps < 2) cps = 2;
    if (cps > k / 8) cps = k / 8;
    o.cps = (uint8_t)cps;
    w16 += (uint32_t)n * (uint32_t)k / 8;  // n * K * 2 bytes / 16
    p->layers[p->nlayers - 1].nops++;
  }
  // One logical [n x k_total] weight matrix (+ 16 bias rows in the folded-bias forward programs), consumed by one or
  // more parts; the parts may sit in consecutive layers (split skip layer, see kMaxTrunkInInb).
  // bias = false: a matrix without bias rows (the hidden parts of the warp stage's split skip layer, whose bias rides with
  // the input part)
  void begin_logical(int n, int k_total, bool bias = true) {
    const int kb = ones_col >= 0 && bias ? 16 : 0;   // bias rows (hn_mlp_program.h: bias folding)
    LogicalOp& l = lg->ops[lg->n++];
    l.w_off16 = w16; l.n = (uint16_t)n; l.k = (uint16_t)(k_total + kb);
    lg_chunks = 0; lg_total = (k_total + kb) / 8;
  }
  void part(int n, int k, Src s, int a_col, int tmem_col, int acc_init) {
    emit(n, k, s, a_col, tmem_col, acc_init, lg_chunks, lg_total);
    lg_chunks += k / 8;
  }
  void bias_part(int n, int tmem_col) {
    if (ones_col < 0) return;
    emit(n, 16, SRC_INB, ones_col, tmem_col, 1, lg_chunks, lg_total);
    p->ops[p->nops - 1].pad = 1;   // marks a bias step
    lg_chunks += 2;
  }
  // the common case: the K range is split over at most two source buffers inside one layer
  void add_op(int n, int k0, Src s0, int a0_col, int k1, Src s1, int a1_col, int tmem_col, int acc_init = 0) {
    begin_logical(n, k0 + k1);
    part(n, k0, s0, a0_col, tmem_col, acc_init);
    if (k1 > 0) part(n, k1, s1, a1_col, tmem_col, 1);
    bias_part(n, tmem_col);
  }
};

// copy of a program without its bias steps (weight offsets are absolute, so the same blob serves both)
void without_bias_steps(const Program& src, Program* dst) {
  memset(dst, 0, sizeof(*dst));
  dst->nlayers = src.nlayers; dst->flags = src.flags;
  for (int li = 0; li < src.nlayers; ++li) {
    Layer L = src.layers[li];
    const int op0 = dst->nops;
    for (int oi = L.op0; oi < L.op0 + L.nops; ++oi)
      if (!src.ops[oi].pad) dst->ops[dst->nops++] = src.ops[oi];
    L.op0 = (uint8_t)op0; L.nops = (uint8_t)(dst->nops - op0);
    dst->layers[li] = L;
  }
}

// layers [l0, l1) of a program as a program of their own (weight offsets are absolute: same blob)
void slice_program(const Program& src, int l0, int l1, Program* dst) {
  memset(dst, 0, sizeof(*dst));
  dst->flags = src.flags;
  for (int li = l0; li < l1; ++li) {
    Layer L = src.layers[li];
    const int op0 = dst->nops;
    for (int oi = L.op0; oi < L.op0 + L.nops; ++oi) dst->ops[dst->nops++] = src.ops[oi];
    L.op0 = (uint8_t)op0;
    dst->layers[dst->nlayers++] = L;
  }
}

// Positional-encoding windows by weight tensor: the source columns [c0, c1) of a tensor that read one encoder's output.
struct WinSeg { int c0, c1; uint8_t win, win_c; };
struct WinLayout {
  uint8_t nseg[HN_NUM_PARAM_TENSORS] = {};
  WinSeg seg[HN_NUM_PARAM_TENSORS][2];
  void add(int param, int c0, int n, PeAlpha a, int C, bool identity) {
    if (n > 0) seg[param][nseg[param]++] = WinSeg{c0, c0 + n, (uint8_t)(1 + a), (uint8_t)(C | (identity ? kWinIdentity : 0))};
  }
  // Splits the source columns [c, c + n) of `param` at its encoder boundaries: piece(offset, count, win, win_c, win_e0).
  template <class F>
  void split(int param, int c, int n, F piece) const {
    int at = 0;
    while (at < n) {
      int end = n;
      uint8_t win = kNoWin, win_c = 0; int e0 = 0;
      for (int i = 0; i < nseg[param]; ++i) {
        const WinSeg& s = seg[param][i];
        if (c + at >= s.c0 && c + at < s.c1) { win = s.win; win_c = s.win_c; e0 = c + at - s.c0; end = std::min(end, s.c1 - c); }
        else if (s.c0 > c + at) end = std::min(end, s.c0 - c);
      }
      piece(at, end - at, win, win_c, e0);
      at = end;
    }
  }
};

// A tensor the configuration does not have carries a negative offset (include/hypernerf_b200.h): its pack blocks are left
// out (the operand image stays zero), its gradient segments are dropped.
struct Packer {
  PackTable* t;
  const int64_t* off;
  const WinLayout* wl = nullptr;   // windowed tables: blocks are split at the encoder boundaries
  int cur = -1;
  void op(const LogicalOp& o) {
    cur = t->nops++;
    PackOp& po = t->ops[cur];
    po.w_off16 = o.w_off16; po.n = o.n; po.k = o.k; po.blk0 = (uint8_t)t->nblocks; po.nblk = 0; po.pad = 0;
  }
  void raw_block(int param, int64_t src_extra, int sn, int sk, int n0, int nn, int k0, int kk, uint8_t win = kNoWin,
                 uint8_t win_c = 0, int win_e0 = 0) {
    PackBlock& b = t->blocks[t->nblocks++];
    b.src = off[param] + src_extra; b.sn = sn; b.sk = sk;
    b.n0 = (uint16_t)n0; b.nn = (uint16_t)nn; b.k0 = (uint16_t)k0; b.kk = (uint16_t)kk;
    b.win = win; b.win_c = win_c; b.win_e0 = (uint16_t)win_e0;
    t->ops[cur].nblk++;
  }
  // src_extra is the block's first source column (row 0): the forward images walk the columns along k (sk == 1), the
  // transposed ones along n (sn == 1)
  void block(int param, int64_t src_extra, int sn, int sk, int n0, int nn, int k0, int kk) {
    if (off[param] < 0 || nn <= 0 || kk <= 0) return;
    if (wl == nullptr || wl->nseg[param] == 0 || sk == kBiasPairStride || (sk != 1 && sn != 1)) {
      raw_block(param, src_extra, sn, sk, n0, nn, k0, kk);
      return;
    }
    const bool along_k = sk == 1;
    wl->split(param, (int)src_extra, along_k ? kk : nn, [&](int o, int cnt, uint8_t win, uint8_t win_c, int e0) {
      if (along_k) raw_block(param, src_extra + o, sn, sk, n0, nn, k0 + o, cnt, win, win_c, e0);
      else raw_block(param, src_extra + o, sn, sk, n0 + o, cnt, k0, kk, win, win_c, e0);
    });
  }
  // bias of output rows [n0, n0 + nn) of the current op into its last two K rows (folded-bias programs)
  void bias_rows(int param, int n0, int nn) {
    const int k0 = t->ops[cur].k - 2;
    block(param, 0, 1, kBiasPairStride, n0, nn, k0, 2);
  }
  void bias(int param, int dst, int cnt) {
    if (off[param] < 0) return;
    BiasBlock& b = t->bias[t->nbias++];
    b.src = off[param]; b.dst = (uint16_t)dst; b.cnt = (uint16_t)cnt; b.pad = 0;
  }
};

}  // namespace

static void build_plan_static(const hn_model_desc& d, ModelPlan* plan);
static void build_tables_static(const int64_t* off, ModelPlan* plan);

void build_plan(const hn_model_desc& d, ModelPlan* plan) {
  memset(plan, 0, sizeof(*plan));
  if (is_static(d)) { build_plan_static(d, plan); return; }
  const Dims m = make_dims(d);
  const SlabMap s = make_slabs(m);
  const bool cond = m.cond_a || m.cond_r;
  plan->dims = m;
  plan->slabs = s;
  int bias_floats = 0;

  // ------------------------------------------------------------------ forward program
  {
    Builder b{&plan->fwd, &plan->fwd_logical};
    b.ones_col = m.ones_col;
    plan->fwd.flags = m.t_in_act ? PF_TIN_ACT : 0;
    int bias = 0;
    if (m.ws_act) {
      // SE3Field + HyperSheetMLP merged to one 192-wide net (SE3 trunk 128 | sheet 64) on the warp-stage vector in ACT
      b.begin_layer(FE_RELU, kWsW, bias, s.x_hws[0], kNone, s.g_hws[0]);
      b.add_op(kWsW, m.KW, SRC_ACT, 0, 0, SRC_ACT, 0, 0);
      bias += kWsW;
      for (int l = 1; l < kWsDepth; ++l) {
        if (l == kSkip + 1) {
          // hidden parts; the FE_SKIPFEED epilogue re-fills ACT[0, KW) with the input vector; then the input part (one
          // block-diagonal 192-row matrix, as layer 0) and the biases on top
          b.begin_layer(FE_SKIPFEED, kWsW, bias, kNone, kNone);
          b.begin_logical(kSe3W, kSe3W, false);
          b.part(kSe3W, kSe3W, SRC_ACT, 0, 0, 0);
          b.begin_logical(kSheetW, kSheetW, false);
          b.part(kSheetW, kSheetW, SRC_ACT, kSe3W, kSe3W, 0);
          b.begin_layer(FE_RELU, kWsW, bias, s.x_hws[l], kNone, s.g_hws[l]);
          b.add_op(kWsW, m.KW, SRC_ACT, 0, 0, SRC_ACT, 0, 0, /*acc_init=*/1);
        } else {
          b.begin_layer(FE_RELU, kWsW, bias, s.x_hws[l], kNone, s.g_hws[l]);
          b.add_op(kSe3W, kSe3W, SRC_ACT, 0, 0, SRC_ACT, 0, 0);
          b.add_op(kSheetW, kSheetW, SRC_ACT, kSe3W, 0, SRC_ACT, 0, kSe3W);
        }
        bias += kWsW;
      }
      // the SE3 trunk's logit layer and the sheet's (64 -> H, accumulator columns [128, 144)): the sheet's must run before
      // the w / v hidden layer, whose 256-wide output overwrites all of ACT
      b.begin_layer(FE_LINSHEET, kSe3W + 16, bias, s.x_se_logit, kNone);
      b.add_op(kSe3W, kSe3W, SRC_ACT, 0, 0, SRC_ACT, 0, 0);
      b.add_op(16, kSheetW, SRC_ACT, kSe3W, 0, SRC_ACT, 0, kSe3W);
      bias += kSe3W + 16;
      b.begin_layer(FE_RELU, 2 * kSe3W, bias, s.x_se_wv, kNone, s.g_se_wv);
      b.add_op(2 * kSe3W, kSe3W, SRC_ACT, 0, 0, SRC_ACT, 0, 0);
      bias += 2 * kSe3W;
      b.begin_layer(FE_WSHEAD, 16, bias, s.x_in_t, kNone);
      b.add_op(16, 2 * kSe3W, SRC_ACT, 0, 0, SRC_ACT, 0, 0);
      bias += 16;
    } else if (m.se3) {
      // SE3Field.warp (warping.py:212-227): trunk on posenc(points) alone, logit layer, merged w / v hidden layer, 6-output head
      b.begin_layer(FE_RELU, kSe3W, bias, s.x_hws[0], kNone, s.g_hws[0]);
      b.add_op(kSe3W, m.KW, SRC_INB, 0, 0, SRC_ACT, 0, 0);
      bias += kSe3W;
      for (int l = 1; l < kWsDepth; ++l) {
        b.begin_layer(FE_RELU, kSe3W, bias, s.x_hws[l], kNone, s.g_hws[l]);
        b.add_op(kSe3W, kSe3W, SRC_ACT, 0, l == kSkip + 1 ? m.KW : 0, SRC_INB, 0, 0);
        bias += kSe3W;
      }
      b.begin_layer(FE_LINEAR, kSe3W, bias, s.x_se_logit, kNone);
      b.add_op(kSe3W, kSe3W, SRC_ACT, 0, 0, SRC_ACT, 0, 0);
      bias += kSe3W;
      b.begin_layer(FE_RELU, 2 * kSe3W, bias, s.x_se_wv, kNone, s.g_se_wv);
      b.add_op(2 * kSe3W, kSe3W, SRC_ACT, 0, 0, SRC_ACT, 0, 0);
      bias += 2 * kSe3W;
      b.begin_layer(FE_WSHEAD, 16, bias, s.x_in_t, kNone);
      b.add_op(16, 2 * kSe3W, SRC_ACT, 0, 0, SRC_ACT, 0, 0);
      bias += 16;
    } else if (!m.nowarp) {
      // warp + sheet, merged to one 192-wide net sharing the input buffer (axis-aligned slicing has no sheet MLP: its
      // part of the operand images stays zero)
      b.begin_layer(FE_RELU, kWsW, bias, s.x_hws[0], kNone, s.g_hws[0]);
      b.add_op(kWsW, m.KW, SRC_INB, 0, 0, SRC_ACT, 0, 0);
      bias += kWsW;
      for (int l = 1; l < kWsDepth; ++l) {
        b.begin_layer(FE_RELU, kWsW, bias, s.x_hws[l], kNone, s.g_hws[l]);
        bool skip = (l == kSkip + 1);
        b.add_op(kWarpW, kWarpW, SRC_ACT, 0, skip ? m.KW : 0, SRC_INB, 0, 0);
        b.add_op(kSheetW, kSheetW, SRC_ACT, kWarpW, skip ? m.KW : 0, SRC_INB, 0, kWarpW);
        bias += kWsW;
      }
      b.begin_layer(FE_WSHEAD, 16, bias, s.x_in_t, kNone);
      b.add_op(16, kWsW, SRC_ACT, 0, 0, SRC_ACT, 0, 0);
      bias += 16;
    }
    const int n_ws_layers = plan->fwd.nlayers;
    // trunk
    const Src tsrc = m.t_in_act ? SRC_ACT : SRC_INB;
    b.begin_layer(FE_RELU, kTrunkW, bias, s.x_t[0], kNone, s.g_t[0]);
    b.add_op(kTrunkW, m.KT, tsrc, 0, 0, SRC_ACT, 0, 0);
    bias += kTrunkW;
    for (int l = 1; l <= kTrunkDepth; ++l) {  // l == kTrunkDepth is the logit layer (ReLU output, modules.py:230)
      const bool skip = (l == kSkip + 1);
      if (skip && m.t_in_act) {
        // hidden part; its epilogue re-fills ACT[0, KT) with the trunk input vector; then the input part on top
        b.begin_layer(FE_SKIPFEED, kTrunkW, bias, kNone, kNone);
        b.begin_logical(kTrunkW, kTrunkW + m.KT);
        b.part(kTrunkW, kTrunkW, SRC_ACT, 0, 0, 0);
        b.begin_layer(FE_RELU, kTrunkW, bias, s.x_t[l], kNone, s.g_t[l]);
        b.part(kTrunkW, m.KT, SRC_ACT, 0, 0, 1);
        b.bias_part(kTrunkW, 0);
      } else {
        b.begin_layer(FE_RELU, kTrunkW, bias, s.x_t[l], kNone, s.g_t[l]);
        b.add_op(kTrunkW, kTrunkW, SRC_ACT, 0, skip ? m.KT : 0, SRC_INB, 0, 0);
      }
      bias += kTrunkW;
    }
    b.begin_layer(FE_BOTT, kRgbW, bias, s.x_bott, kNone);
    b.add_op(kRgbW, kTrunkW, SRC_ACT, 0, 0, SRC_ACT, 0, 0);
    bias += kRgbW;
    b.begin_layer(FE_RGB0A, m.n_rgb0a, bias, s.x_r[0], kNone, s.g_r[0]);
    b.add_op(m.n_rgb0a, kRgbW, SRC_ACT, 0, m.KV, SRC_INB, 0, 0);
    bias += m.n_rgb0a;
    for (int l = 1; l < kRgbDepth; ++l) {
      b.begin_layer(FE_RELU, kRgbW, bias, s.x_r[l], kNone, s.g_r[l]);
      b.add_op(kRgbW, kRgbW, SRC_ACT, 0, 0, SRC_ACT, 0, 0);
      bias += kRgbW;
    }
    b.begin_layer(FE_RGBHEAD, 16, bias, kNone, kNone);
    b.add_op(16, kRgbW, SRC_ACT, 0, 0, SRC_ACT, 0, 0);
    bias += 16;
    bias_floats = bias;
    plan->layout.fwd_off = 0;
    plan->layout.bwd_off = (int64_t)b.w16 * 16;
    without_bias_steps(plan->fwd, &plan->fwd_train);
    // trunk-only: everything after the warp / sheet head (without warp that is the whole program)
    slice_program(plan->fwd, n_ws_layers, plan->fwd.nlayers, &plan->fwd_trunk);
    slice_program(plan->fwd_train, n_ws_layers, plan->fwd_train.nlayers, &plan->fwd_trunk_train);
    // warp-stage-only: the complementary slice, up to and including the warp / sheet head
    if (!m.nowarp) {
      slice_program(plan->fwd, 0, n_ws_layers, &plan->fwd_warp);
      slice_program(plan->fwd_train, 0, n_ws_layers, &plan->fwd_warp_train);
      plan->fwd_warp.flags |= PF_WARP_ONLY;
      plan->fwd_warp_train.flags |= PF_WARP_ONLY;
      if (!m.se3) {
        plan->fwd_warp_tangent = plan->fwd_warp_train;
        plan->fwd_warp_tangent.flags |= PF_TANGENT;
        for (int l = 0; l < plan->fwd_warp_tangent.nlayers; ++l) {
          Layer& L = plan->fwd_warp_tangent.layers[l];
          L.epi = L.epi == FE_RELU ? FE_TANGENT : FE_JACHEAD;
        }
      }
    }
  }
  // ------------------------------------------------------------------ backward-data program
  {
    Builder b{&plan->bwd, &plan->bwd_logical};
    // D0: rgb head^T.  A = dY_rgbhead (16 cols, written by the prologue)
    b.begin_layer(BE_MASK, kRgbW, 0, s.d_r[3], s.x_r[3], s.g_r[3]);
    b.add_op(kRgbW, 16, SRC_ACT, 0, 0, SRC_ACT, 0, 0);
    // D1..D3: rgb3^T, rgb2^T, rgb1^T
    for (int l = kRgbDepth - 1; l >= 1; --l) {
      bool last = (l == 1);
      b.begin_layer(last ? BE_RGB1 : BE_MASK, kRgbW, 0, last ? s.d_rgb0a : s.d_r[l - 1], s.x_r[l - 1], s.g_r[l - 1]);
      b.add_op(kRgbW, kRgbW, SRC_ACT, 0, 0, SRC_ACT, 0, 0);
    }
    // D4: (rgb0 | alpha)^T -> bottleneck gradient (no activation on the bottleneck, modules.py:232,277); with template
    // conditioning also the gradient of the GLO columns of the view vector, parked in TMEM cols [128, 144)
    b.begin_layer(cond ? BE_LINCOND : BE_LINEAR, kRgbW, 0, s.d_bott, kNone);
    b.add_op(kRgbW, m.n_rgb0a, SRC_ACT, 0, 0, SRC_ACT, 0, 0);
    if (cond) b.add_op(16, m.n_rgb0a, SRC_ACT, 0, 0, SRC_ACT, 0, kRgbW);
    // D5: bottleneck^T, gated by the trunk output ReLU
    b.begin_layer(BE_MASK, kTrunkW, 0, s.d_t[kTrunkDepth], s.x_t[kTrunkDepth], s.g_t[kTrunkDepth]);
    b.add_op(kTrunkW, kRgbW, SRC_ACT, 0, 0, SRC_ACT, 0, 0);
    // trunk layers l = 8 (logit) .. 1: gradient w.r.t. h_{l-1}
    for (int l = kTrunkDepth; l >= 1; --l) {
      if (l == kSkip + 1) {
        // input part of the skip layer first (pulled back through the posenc chain rule by the epilogue), then the hidden part
        b.begin_layer(BE_SKIPSTORE, m.KT, 0, kNone, kNone);
        b.add_op(m.KT, kTrunkW, SRC_ACT, 0, 0, SRC_ACT, 0, 0);
      }
      b.begin_layer(BE_MASK, kTrunkW, 0, s.d_t[l - 1], s.x_t[l - 1], s.g_t[l - 1]);
      b.add_op(kTrunkW, kTrunkW, SRC_ACT, 0, 0, SRC_ACT, 0, 0);
    }
    // trunk layer 0^T -> gradient of the trunk input features -> chain rule through posenc
    b.begin_layer(BE_TRUNKIN, m.KT, 0, m.nowarp ? kNone : s.d_wshead, kNone);
    b.add_op(m.KT, kTrunkW, SRC_ACT, 0, 0, SRC_ACT, 0, 0);
    const int n_trunk_layers = plan->bwd.nlayers;
    if (m.se3) {
      // head^T: A = d(w, v) (16 columns, written by BE_TRUNKIN's exp-map chain rule), gated by the w / v hidden ReLUs
      b.begin_layer(BE_MASK, 2 * kSe3W, 0, s.d_se_wv, s.x_se_wv, s.g_se_wv);
      b.add_op(2 * kSe3W, 16, SRC_ACT, 0, 0, SRC_ACT, 0, 0);
      // (w hidden | v hidden)^T -> gradient of the logit layer's output (no activation); with the sheet, the epilogue also
      // writes the sheet head's dY into ACT[128, 144)
      b.begin_layer(m.ws_act ? BE_LINSHEET : BE_LINEAR, kSe3W, 0, s.d_se_logit, kNone);
      b.add_op(kSe3W, 2 * kSe3W, SRC_ACT, 0, 0, SRC_ACT, 0, 0);
      if (m.ws_act) {
        // (SE3 logit | sheet logit)^T, gated by layer 5's ReLUs, then layers 5..1 as in the translation configurations (the
        // sample point takes no gradient, the GLO columns of the sheet's inputs go to the table)
        b.begin_layer(BE_MASK, kWsW, 0, s.d_ws[kWsDepth - 1], s.x_hws[kWsDepth - 1], s.g_hws[kWsDepth - 1]);
        b.add_op(kSe3W, kSe3W, SRC_ACT, 0, 0, SRC_ACT, 0, 0);
        b.add_op(kSheetW, 16, SRC_ACT, kSe3W, 0, SRC_ACT, 0, kSe3W);
        for (int l = kWsDepth - 1; l >= 1; --l) {
          b.begin_layer(BE_MASK, kWsW, 0, s.d_ws[l - 1], s.x_hws[l - 1], s.g_hws[l - 1]);
          if (l == kSkip + 1)  // GLO columns of the sheet's skip input, parked in TMEM cols [192, 208)
            b.add_op(16, kWsW, SRC_ACT, 0, 0, SRC_ACT, 0, kWsW);
          b.add_op(kSe3W, kSe3W, SRC_ACT, 0, 0, SRC_ACT, 0, 0);
          b.add_op(kSheetW, kSheetW, SRC_ACT, kSe3W, 0, SRC_ACT, 0, kSe3W);
        }
        b.begin_layer(BE_GLO, 16, 0, kNone, kNone);
        b.add_op(16, kWsW, SRC_ACT, 0, 0, SRC_ACT, 0, kWsW, /*acc_init=*/1);
      } else {
        // logit^T, then trunk layers 5..1 (the skip layer's input part is posenc(points): no gradient wanted)
        for (int l = kWsDepth; l >= 1; --l) {
          b.begin_layer(BE_MASK, kSe3W, 0, s.d_ws[l - 1], s.x_hws[l - 1], s.g_hws[l - 1]);
          b.add_op(kSe3W, kSe3W, SRC_ACT, 0, 0, SRC_ACT, 0, 0);
        }
      }
    } else if (!m.nowarp) {
      // warp/sheet head^T
      b.begin_layer(BE_MASK, kWsW, 0, s.d_ws[kWsDepth - 1], s.x_hws[kWsDepth - 1], s.g_hws[kWsDepth - 1]);
      b.add_op(kWsW, 16, SRC_ACT, 0, 0, SRC_ACT, 0, 0);
      for (int l = kWsDepth - 1; l >= 1; --l) {
        b.begin_layer(BE_MASK, kWsW, 0, s.d_ws[l - 1], s.x_hws[l - 1], s.g_hws[l - 1]);
        if (l == kSkip + 1)  // GLO columns of the skip input, parked in TMEM cols [192,208)
          b.add_op(16, kWsW, SRC_ACT, 0, 0, SRC_ACT, 0, kWsW);
        b.add_op(kWarpW, kWarpW, SRC_ACT, 0, 0, SRC_ACT, 0, 0);
        b.add_op(kSheetW, kSheetW, SRC_ACT, kWarpW, 0, SRC_ACT, 0, kWarpW);
      }
      // GLO columns of layer 0, accumulated on top
      b.begin_layer(BE_GLO, 16, 0, kNone, kNone);
      b.add_op(16, kWsW, SRC_ACT, 0, 0, SRC_ACT, 0, kWsW, /*acc_init=*/1);
    }
    plan->layout.bias_off = plan->layout.bwd_off + (int64_t)b.w16 * 16;
    // trunk-only: up to and including the trunk-input layer (BE_TRUNKIN), whose epilogue then emits d(warped point)
    slice_program(plan->bwd, 0, n_trunk_layers, &plan->bwd_trunk);
    // warp-stage-only: from the head^T layer on (the prologue seeds its A operand from g_warped)
    if (!m.nowarp) {
      slice_program(plan->bwd, n_trunk_layers, plan->bwd.nlayers, &plan->bwd_warp);
      plan->bwd_warp.flags |= PF_WARP_ONLY;
    }
  }
  PlanInfo& I = plan->info;
  I.glo_param = m.nowarp ? (cond ? P_COND_GLO : -1) : P_GLO;
  I.glo_floats = I.glo_param >= 0 ? d.num_embeddings * m.G : 0;
  plan->layout.glo_off = plan->layout.bias_off + (int64_t)bias_floats * 4;
  plan->layout.glo_off = (plan->layout.glo_off + 15) / 16 * 16;
  plan->layout.total = plan->layout.glo_off + (int64_t)I.glo_floats * 4;
  plan->layout.total = (plan->layout.total + 255) / 256 * 256;
  I.x_total = s.x_total; I.d_total = s.d_total; I.g_total = s.g_total;
  I.x_in0 = s.x_in_ws; I.x_in_t = s.x_in_t; I.x_in_v = s.x_in_v;
  I.d_rgbhead = s.d_rgbhead; I.d_sigma = kNone;
  if (!m.nowarp) { I.x_warp = s.x_in_t; I.d_warp = s.d_t[0]; I.g_warp = s.g_t[0]; }
  I.n_params = HN_NUM_PARAM_TENSORS;
}

void build_tables(const hn_model_desc& d, int level, const int64_t* off, bool windowed, ModelPlan* plan) {
  if (is_static(d)) { build_tables_static(off, plan); return; }
  const Dims& m = plan->dims;
  const SlabMap& s = plan->slabs;
  const bool cond = m.cond_a || m.cond_r;
  // ------------------------------------------------------------------ positional-encoding windows
  // (reference column space; the skip layers read [hidden | input vector])
  WinLayout wl;
  if (m.se3) {
    wl.add(P_WARP_W(0), 0, m.pe_w, PE_WARP, 3, false);                 // posenc(points, 0, 8): bands of 6, no identity
    wl.add(P_WARP_W(kSkip + 1), kSe3W, m.pe_w, PE_WARP, 3, false);
    if (m.ws_act) {
      wl.add(P_SHEET_W(0), 0, m.pe_s, PE_SHEET, 3, true);              // posenc_orig(points, 7)
      wl.add(P_SHEET_W(kSkip + 1), kSheetW, m.pe_s, PE_SHEET, 3, true);
    }
  } else if (!m.nowarp) {
    wl.add(P_WARP_W(0), 0, m.pe_w, PE_WARP, 3, true);                  // posenc_orig(points, 10)
    wl.add(P_WARP_W(kSkip + 1), kWarpW, m.pe_w, PE_WARP, 3, true);
    wl.add(P_SHEET_W(0), 0, m.pe_s, PE_SHEET, 3, true);                // posenc_orig(points, 7)
    wl.add(P_SHEET_W(kSkip + 1), kSheetW, m.pe_s, PE_SHEET, 3, true);
  }
  for (int l : {0, kSkip + 1}) {                                       // posenc_orig(xyz) | posenc_orig(hyper point)
    const int c = l == 0 ? 0 : kTrunkW;
    wl.add(P_TRUNK_W(level, l), c, m.pe_x, PE_NERF, 3, true);
    wl.add(P_TRUNK_W(level, l), c + m.pe_x, m.pe_h, PE_HYPER, m.H, true);
  }
  // ------------------------------------------------------------------ pack table
  PackTable& t = plan->pack;
  memset(&t, 0, sizeof(t));
  Packer pk{&t, off, windowed ? &wl : nullptr};
  const LogicalOps& F = plan->fwd_logical;
  int oi = 0;
  const int ldw5 = kWarpW + m.in_w, lds5 = kSheetW + m.in_s;
  // rgb layer 0 reads [bottleneck | view PE (pe_v) | GLO (rgb condition)], the alpha head [bottleneck | GLO (alpha condition)]
  // (modules.py:283,292); inside the operand the view vector is [PE padded to 40 | GLO] (hn_mlp_program.h: kViewCondCol)
  const int ld_rgb0 = kRgbW + m.pe_v + (m.cond_r ? m.G : 0), ld_alpha = kRgbW + (m.cond_a ? m.G : 0);
  const int k_cond = kRgbW + kViewCondCol;
  const int ld_se5 = kSe3W + m.in_w;
  if (m.ws_act) {
    // warp-stage vector: [posenc(points, 0, 8) | posenc_orig(points, 7) | GLO]; the sheet reads it from column pe_w on
    pk.op(F.ops[oi++]);  // layer 0: rows [0, 128) SE3 trunk, rows [128, 192) sheet
    pk.block(P_WARP_W(0), 0, m.in_w, 1, 0, kSe3W, 0, m.in_w);
    pk.block(P_SHEET_W(0), 0, m.in_s, 1, kSe3W, kSheetW, m.pe_w, m.in_s);
    pk.bias_rows(P_WARP_B(0), 0, kSe3W);
    pk.bias_rows(P_SHEET_B(0), kSe3W, kSheetW);
    for (int l = 1; l < kWsDepth; ++l) {
      if (l == kSkip + 1) {   // hidden parts, then the input part of both nets with their biases
        pk.op(F.ops[oi++]);
        pk.block(P_WARP_W(l), 0, ld_se5, 1, 0, kSe3W, 0, kSe3W);
        pk.op(F.ops[oi++]);
        pk.block(P_SHEET_W(l), 0, lds5, 1, 0, kSheetW, 0, kSheetW);
        pk.op(F.ops[oi++]);
        pk.block(P_WARP_W(l), kSe3W, ld_se5, 1, 0, kSe3W, 0, m.in_w);
        pk.block(P_SHEET_W(l), kSheetW, lds5, 1, kSe3W, kSheetW, m.pe_w, m.in_s);
        pk.bias_rows(P_WARP_B(l), 0, kSe3W);
        pk.bias_rows(P_SHEET_B(l), kSe3W, kSheetW);
      } else {
        pk.op(F.ops[oi++]);
        pk.block(P_WARP_W(l), 0, kSe3W, 1, 0, kSe3W, 0, kSe3W);
        pk.bias_rows(P_WARP_B(l), 0, kSe3W);
        pk.op(F.ops[oi++]);
        pk.block(P_SHEET_W(l), 0, kSheetW, 1, 0, kSheetW, 0, kSheetW);
        pk.bias_rows(P_SHEET_B(l), 0, kSheetW);
      }
    }
    pk.op(F.ops[oi++]);  // SE3 logit layer
    pk.block(P_WARP_W(kWsDepth), 0, kSe3W, 1, 0, kSe3W, 0, kSe3W);
    pk.bias_rows(P_WARP_B(kWsDepth), 0, kSe3W);
    pk.op(F.ops[oi++]);  // sheet logit layer: rows 0..H-1
    pk.block(P_SHEET_W(kWsDepth), 0, kSheetW, 1, 0, m.H, 0, kSheetW);
    pk.bias_rows(P_SHEET_B(kWsDepth), 0, m.H);
  } else if (m.se3) {
    pk.op(F.ops[oi++]);
    pk.block(P_WARP_W(0), 0, m.in_w, 1, 0, kSe3W, 0, m.in_w);
    pk.bias_rows(P_WARP_B(0), 0, kSe3W);
    for (int l = 1; l <= kWsDepth; ++l) {   // l == kWsDepth: the trunk's logit layer
      const int ld = l == kSkip + 1 ? ld_se5 : kSe3W;
      pk.op(F.ops[oi++]);
      pk.block(P_WARP_W(l), 0, ld, 1, 0, kSe3W, 0, ld);
      pk.bias_rows(P_WARP_B(l), 0, kSe3W);
    }
  }
  if (m.se3) {
    pk.op(F.ops[oi++]);  // rows [0, 128) w_net.linears.0, [128, 256) v_net.linears.0
    pk.block(P_SE3_W(SE3_W_HID), 0, kSe3W, 1, 0, kSe3W, 0, kSe3W);
    pk.block(P_SE3_W(SE3_V_HID), 0, kSe3W, 1, kSe3W, kSe3W, 0, kSe3W);
    pk.bias_rows(P_SE3_B(SE3_W_HID), 0, kSe3W);
    pk.bias_rows(P_SE3_B(SE3_V_HID), kSe3W, kSe3W);
    pk.op(F.ops[oi++]);  // head: rows 0..2 = w_net.logit_layer on the w hidden columns, rows 3..5 = v_net.logit_layer on the v ones
    pk.block(P_SE3_W(SE3_W_OUT), 0, kSe3W, 1, 0, 3, 0, kSe3W);
    pk.block(P_SE3_W(SE3_V_OUT), 0, kSe3W, 1, 3, 3, kSe3W, kSe3W);
    pk.bias_rows(P_SE3_B(SE3_W_OUT), 0, 3);
    pk.bias_rows(P_SE3_B(SE3_V_OUT), 3, 3);
  } else if (!m.nowarp) {
    // fwd ws0
    pk.op(F.ops[oi++]);
    pk.block(P_WARP_W(0), 0, m.in_w, 1, 0, kWarpW, 0, m.in_w);
    pk.block(P_SHEET_W(0), 0, m.in_s, 1, kWarpW, kSheetW, 0, m.pe_s);
    pk.block(P_SHEET_W(0), m.pe_s, m.in_s, 1, kWarpW, kSheetW, m.pe_w, m.G);
    pk.bias_rows(P_WARP_B(0), 0, kWarpW);
    pk.bias_rows(P_SHEET_B(0), kWarpW, kSheetW);
    for (int l = 1; l < kWsDepth; ++l) {
      bool skip = (l == kSkip + 1);
      pk.op(F.ops[oi++]);
      pk.block(P_WARP_W(l), 0, skip ? ldw5 : kWarpW, 1, 0, kWarpW, 0, skip ? ldw5 : kWarpW);
      pk.bias_rows(P_WARP_B(l), 0, kWarpW);
      pk.op(F.ops[oi++]);
      if (!skip) {
        pk.block(P_SHEET_W(l), 0, kSheetW, 1, 0, kSheetW, 0, kSheetW);
      } else {
        pk.block(P_SHEET_W(l), 0, lds5, 1, 0, kSheetW, 0, kSheetW + m.pe_s);
        pk.block(P_SHEET_W(l), kSheetW + m.pe_s, lds5, 1, 0, kSheetW, kSheetW + m.pe_w, m.G);
      }
      pk.bias_rows(P_SHEET_B(l), 0, kSheetW);
    }
    pk.op(F.ops[oi++]);  // ws head: rows 0..2 warp logit, rows 3..3+H-1 sheet logit
    pk.block(P_WARP_W(kWsDepth), 0, kWarpW, 1, 0, 3, 0, kWarpW);
    pk.block(P_SHEET_W(kWsDepth), 0, kSheetW, 1, 3, m.H, kWarpW, kSheetW);
    pk.bias_rows(P_WARP_B(kWsDepth), 0, 3);
    pk.bias_rows(P_SHEET_B(kWsDepth), 3, m.H);
  }
  pk.op(F.ops[oi++]);  // trunk 0
  pk.block(P_TRUNK_W(level, 0), 0, m.in_t, 1, 0, kTrunkW, 0, m.in_t);
  pk.bias_rows(P_TRUNK_B(level, 0), 0, kTrunkW);
  for (int l = 1; l <= kTrunkDepth; ++l) {
    int ld = (l == kSkip + 1) ? kTrunkW + m.in_t : kTrunkW;
    pk.op(F.ops[oi++]);
    pk.block(P_TRUNK_W(level, l), 0, ld, 1, 0, kTrunkW, 0, ld);
    pk.bias_rows(P_TRUNK_B(level, l), 0, kTrunkW);
  }
  pk.op(F.ops[oi++]);  // bottleneck
  pk.block(P_BOTT_W(level), 0, kTrunkW, 1, 0, kRgbW, 0, kTrunkW);
  pk.bias_rows(P_BOTT_B(level), 0, kRgbW);
  pk.op(F.ops[oi++]);  // rgb0 | alpha
  pk.block(P_RGB_W(level, 0), 0, ld_rgb0, 1, 0, kRgbW, 0, kRgbW + m.pe_v);
  if (m.cond_r) pk.block(P_RGB_W(level, 0), kRgbW + m.pe_v, ld_rgb0, 1, 0, kRgbW, k_cond, m.G);
  pk.block(P_ALPHA_W(level), 0, ld_alpha, 1, kRgbW, 1, 0, kRgbW);
  if (m.cond_a) pk.block(P_ALPHA_W(level), kRgbW, ld_alpha, 1, kRgbW, 1, k_cond, m.G);
  pk.bias_rows(P_RGB_B(level, 0), 0, kRgbW);
  pk.bias_rows(P_ALPHA_B(level), kRgbW, 1);
  for (int l = 1; l < kRgbDepth; ++l) {
    pk.op(F.ops[oi++]);
    pk.block(P_RGB_W(level, l), 0, kRgbW, 1, 0, kRgbW, 0, kRgbW);
    pk.bias_rows(P_RGB_B(level, l), 0, kRgbW);
  }
  pk.op(F.ops[oi++]);  // rgb head
  pk.block(P_RGB_W(level, kRgbDepth), 0, kRgbW, 1, 0, 3, 0, kRgbW);
  pk.bias_rows(P_RGB_B(level, kRgbDepth), 0, 3);

  // bwd: dest(n = input feature, k = output feature) = W[k][n]  -> sn = 1, sk = ld
  const LogicalOps& Bp = plan->bwd_logical;
  const uint32_t bwd16 = (uint32_t)(plan->layout.bwd_off / 16);
  oi = 0;
  auto bop = [&](void) { LogicalOp o = Bp.ops[oi++]; o.w_off16 += bwd16; pk.op(o); };
  bop();  // D0 rgb head^T: n < 128, k < 3
  pk.block(P_RGB_W(level, kRgbDepth), 0, 1, kRgbW, 0, kRgbW, 0, 3);
  for (int l = kRgbDepth - 1; l >= 1; --l) {
    bop();
    pk.block(P_RGB_W(level, l), 0, 1, kRgbW, 0, kRgbW, 0, kRgbW);
  }
  bop();  // D4
  pk.block(P_RGB_W(level, 0), 0, 1, ld_rgb0, 0, kRgbW, 0, kRgbW);
  pk.block(P_ALPHA_W(level), 0, 1, ld_alpha, 0, kRgbW, kRgbW, 1);
  if (cond) {  // GLO condition columns: dest(g, k < 128) = Wrgb0[k][128 + pe_v + g], dest(g, 128) = Walpha[0][128 + g]
    bop();
    if (m.cond_r) pk.block(P_RGB_W(level, 0), kRgbW + m.pe_v, 1, ld_rgb0, 0, m.G, 0, kRgbW);
    if (m.cond_a) pk.block(P_ALPHA_W(level), kRgbW, 1, ld_alpha, 0, m.G, kRgbW, 1);
  }
  bop();  // D5 bottleneck^T: n < 256, k < 128
  pk.block(P_BOTT_W(level), 0, 1, kTrunkW, 0, kTrunkW, 0, kRgbW);
  for (int l = kTrunkDepth; l >= 1; --l) {
    int ld = (l == kSkip + 1) ? kTrunkW + m.in_t : kTrunkW;
    if (l == kSkip + 1) {
      bop();
      pk.block(P_TRUNK_W(level, l), kTrunkW, 1, ld, 0, m.in_t, 0, kTrunkW);
    }
    bop();
    pk.block(P_TRUNK_W(level, l), 0, 1, ld, 0, kTrunkW, 0, kTrunkW);
  }
  bop();  // trunk 0^T
  pk.block(P_TRUNK_W(level, 0), 0, 1, m.in_t, 0, m.in_t, 0, kTrunkW);
  if (m.se3) {
    bop();  // head^T: n < 128 <- w_net.logit_layer (k < 3); n = 128 + j <- v_net.logit_layer (k = 3 + i)
    pk.block(P_SE3_W(SE3_W_OUT), 0, 1, kSe3W, 0, kSe3W, 0, 3);
    pk.block(P_SE3_W(SE3_V_OUT), 0, 1, kSe3W, kSe3W, kSe3W, 3, 3);
    bop();  // (w hidden | v hidden)^T: dest(n, k < 128) = Wwh[k][n], dest(n, 128 + k) = Wvh[k][n]
    pk.block(P_SE3_W(SE3_W_HID), 0, 1, kSe3W, 0, kSe3W, 0, kSe3W);
    pk.block(P_SE3_W(SE3_V_HID), 0, 1, kSe3W, 0, kSe3W, kSe3W, kSe3W);
    if (m.ws_act) {
      bop();  // SE3 logit^T
      pk.block(P_WARP_W(kWsDepth), 0, 1, kSe3W, 0, kSe3W, 0, kSe3W);
      bop();  // sheet logit^T: dest(j < 64, h < H) = sheetW6[h][j]
      pk.block(P_SHEET_W(kWsDepth), 0, 1, kSheetW, 0, kSheetW, 0, m.H);
      for (int l = kWsDepth - 1; l >= 1; --l) {
        const bool skip = (l == kSkip + 1);
        if (skip) {  // GLO columns of the sheet's skip input: dest(g, 128 + j) = sheetW5[j][64 + pe_s + g]
          bop();
          pk.block(P_SHEET_W(l), kSheetW + m.pe_s, 1, lds5, 0, m.G, kSe3W, kSheetW);
        }
        bop();
        pk.block(P_WARP_W(l), 0, 1, skip ? ld_se5 : kSe3W, 0, kSe3W, 0, kSe3W);
        bop();
        pk.block(P_SHEET_W(l), 0, 1, skip ? lds5 : kSheetW, 0, kSheetW, 0, kSheetW);
      }
      bop();  // GLO columns of the sheet's layer 0
      pk.block(P_SHEET_W(0), m.pe_s, 1, m.in_s, 0, m.G, kSe3W, kSheetW);
    } else {
      for (int l = kWsDepth; l >= 1; --l) {
        bop();
        pk.block(P_WARP_W(l), 0, 1, l == kSkip + 1 ? ld_se5 : kSe3W, 0, kSe3W, 0, kSe3W);
      }
    }
  } else if (!m.nowarp) {
    bop();  // ws head^T: n < 128 <- warp logit (k < 3); n = 128 + j <- sheet logit (k = 3 + h)
    pk.block(P_WARP_W(kWsDepth), 0, 1, kWarpW, 0, kWarpW, 0, 3);
    pk.block(P_SHEET_W(kWsDepth), 0, 1, kSheetW, kWarpW, kSheetW, 3, m.H);
    for (int l = kWsDepth - 1; l >= 1; --l) {
      bool skip = (l == kSkip + 1);
      if (skip) {  // GLO columns: dest(g, k<128) = warpW5[k][128 + pe_w + g]; dest(g, 128 + j) = sheetW5[j][64 + pe_s + g]
        bop();
        pk.block(P_WARP_W(l), kWarpW + m.pe_w, 1, ldw5, 0, m.G, 0, kWarpW);
        pk.block(P_SHEET_W(l), kSheetW + m.pe_s, 1, lds5, 0, m.G, kWarpW, kSheetW);
      }
      bop();
      pk.block(P_WARP_W(l), 0, 1, skip ? ldw5 : kWarpW, 0, kWarpW, 0, kWarpW);
      bop();
      pk.block(P_SHEET_W(l), 0, 1, skip ? lds5 : kSheetW, 0, kSheetW, 0, kSheetW);
    }
    bop();  // GLO columns of layer 0
    pk.block(P_WARP_W(0), m.pe_w, 1, m.in_w, 0, m.G, 0, kWarpW);
    pk.block(P_SHEET_W(0), m.pe_s, 1, m.in_s, 0, m.G, kWarpW, kSheetW);
  }

  // biases, in forward layer order
  int bo = 0;
  if (m.ws_act) {
    for (int l = 0; l < kWsDepth; ++l) {
      pk.bias(P_WARP_B(l), bo, kSe3W);
      pk.bias(P_SHEET_B(l), bo + kSe3W, kSheetW);
      bo += kWsW;
    }
    pk.bias(P_WARP_B(kWsDepth), bo, kSe3W);
    pk.bias(P_SHEET_B(kWsDepth), bo + kSe3W, m.H);
    bo += kSe3W + 16;
  }
  if (m.se3) {
    if (!m.ws_act)
      for (int l = 0; l <= kWsDepth; ++l) { pk.bias(P_WARP_B(l), bo, kSe3W); bo += kSe3W; }
    pk.bias(P_SE3_B(SE3_W_HID), bo, kSe3W);
    pk.bias(P_SE3_B(SE3_V_HID), bo + kSe3W, kSe3W);
    bo += 2 * kSe3W;
    pk.bias(P_SE3_B(SE3_W_OUT), bo, 3);
    pk.bias(P_SE3_B(SE3_V_OUT), bo + 3, 3);
    bo += 16;
  } else if (!m.nowarp) {
    for (int l = 0; l < kWsDepth; ++l) {
      pk.bias(P_WARP_B(l), bo, kWarpW);
      pk.bias(P_SHEET_B(l), bo + kWarpW, kSheetW);
      bo += kWsW;
    }
    pk.bias(P_WARP_B(kWsDepth), bo, 3);
    pk.bias(P_SHEET_B(kWsDepth), bo + 3, m.H);
    bo += 16;
  }
  for (int l = 0; l <= kTrunkDepth; ++l) { pk.bias(P_TRUNK_B(level, l), bo, kTrunkW); bo += kTrunkW; }
  pk.bias(P_BOTT_B(level), bo, kRgbW); bo += kRgbW;
  pk.bias(P_RGB_B(level, 0), bo, kRgbW);
  pk.bias(P_ALPHA_B(level), bo + kRgbW, 1);
  bo += m.n_rgb0a;
  for (int l = 1; l < kRgbDepth; ++l) { pk.bias(P_RGB_B(level, l), bo, kRgbW); bo += kRgbW; }
  pk.bias(P_RGB_B(level, kRgbDepth), bo, 3);
  bo += 16;
  t.bias_floats = bo;

  // ------------------------------------------------------------------ weight-gradient jobs
  WgradTable& w = plan->wgrad;
  memset(&w, 0, sizeof(w));
  auto job = [&](int dy_chunk, int dy_cols, int x0_chunk, int x0_cols, int x1_chunk, int x1_cols) -> WgradJob& {
    WgradJob& j = w.jobs[w.njobs++];
    j.dy_chunk = (uint16_t)dy_chunk; j.dy_nchunks = (uint16_t)(dy_cols / 8);
    j.x0_chunk = (uint16_t)x0_chunk; j.x0_nchunks = (uint16_t)(x0_cols / 8);
    j.x1_chunk = (uint16_t)x1_chunk; j.x1_nchunks = (uint16_t)(x1_cols / 8);
    j.mblocks = (uint8_t)((dy_cols + 127) / 128);
    return j;
  };
  // `extra` is the segment's first source column; windowed tables split it at the encoder boundaries (<= 3 pieces)
  auto flush = [&](WgradJob& j, int param, int64_t extra, int ld, int row0, int nrows, int col0, int ncols) {
    if (off[param] < 0 || nrows <= 0 || ncols <= 0) return;
    auto piece = [&](int o, int cnt, uint8_t win, uint8_t win_c, int e0) {
      FlushSeg& f = j.flush[j.nflush++];
      f.dst = off[param] + extra + o; f.ld = ld; f.row0 = (uint16_t)row0; f.nrows = (uint16_t)nrows;
      f.col0 = (uint16_t)(col0 + o); f.ncols = (uint16_t)cnt;
      f.win = win; f.win_c = win_c; f.win_e0 = (uint16_t)e0;
    };
    if (windowed) wl.split(param, (int)extra, ncols, piece);
    else piece(0, ncols, kNoWin, 0, 0);
  };
  auto bseg = [&](WgradJob& j, int param, int col0, int ncols) {
    if (off[param] < 0 || ncols <= 0) return;
    BiasSeg& b = j.bias[j.nbias++];
    b.dst = off[param]; b.col0 = (uint16_t)col0; b.ncols = (uint16_t)ncols; b.pad = 0;
  };
  // a job none of whose outputs exists (the sheet MLP with axis-aligned slicing) is dropped again
  auto keep = [&](WgradJob& j) { if (j.nflush == 0 && j.nbias == 0) { memset(&j, 0, sizeof(j)); --w.njobs; } };
  if (m.se3) {
    {
      WgradJob& j = job(s.d_ws[0], kSe3W, s.x_in_ws, m.KW, 0, 0);
      flush(j, P_WARP_W(0), 0, m.in_w, 0, kSe3W, 0, m.in_w);
      bseg(j, P_WARP_B(0), 0, kSe3W);
      if (m.ws_act) {   // the sheet reads the warp-stage vector from column pe_w on
        WgradJob& k = job(s.d_ws[0] + kSe3W / 8, kSheetW, s.x_in_ws, m.KW, 0, 0);
        flush(k, P_SHEET_W(0), 0, m.in_s, 0, kSheetW, m.pe_w, m.in_s);
        bseg(k, P_SHEET_B(0), 0, kSheetW);
      }
    }
    for (int l = 1; l < kWsDepth; ++l) {
      const bool skip = (l == kSkip + 1);
      WgradJob& j = job(s.d_ws[l], kSe3W, s.x_hws[l - 1], kSe3W, s.x_in_ws, skip ? m.KW : 0);
      flush(j, P_WARP_W(l), 0, skip ? ld_se5 : kSe3W, 0, kSe3W, 0, skip ? ld_se5 : kSe3W);
      bseg(j, P_WARP_B(l), 0, kSe3W);
      if (m.ws_act) {
        WgradJob& k = job(s.d_ws[l] + kSe3W / 8, kSheetW, s.x_hws[l - 1] + kSe3W / 8, kSheetW, s.x_in_ws, skip ? m.KW : 0);
        flush(k, P_SHEET_W(l), 0, skip ? lds5 : kSheetW, 0, kSheetW, 0, kSheetW);
        if (skip) flush(k, P_SHEET_W(l), kSheetW, lds5, 0, kSheetW, kSheetW + m.pe_w, m.in_s);
        bseg(k, P_SHEET_B(l), 0, kSheetW);
      }
    }
    if (m.ws_act) {
      WgradJob& j = job(s.d_sheethead, 16, s.x_hws[kWsDepth - 1] + kSe3W / 8, kSheetW, 0, 0);
      flush(j, P_SHEET_W(kWsDepth), 0, kSheetW, 0, m.H, 0, kSheetW);
      bseg(j, P_SHEET_B(kWsDepth), 0, m.H);
    }
    {
      WgradJob& j = job(s.d_se_logit, kSe3W, s.x_hws[kWsDepth - 1], kSe3W, 0, 0);
      flush(j, P_WARP_W(kWsDepth), 0, kSe3W, 0, kSe3W, 0, kSe3W);
      bseg(j, P_WARP_B(kWsDepth), 0, kSe3W);
    }
    {
      WgradJob& j = job(s.d_se_wv, 2 * kSe3W, s.x_se_logit, kSe3W, 0, 0);
      flush(j, P_SE3_W(SE3_W_HID), 0, kSe3W, 0, kSe3W, 0, kSe3W);
      flush(j, P_SE3_W(SE3_V_HID), 0, kSe3W, kSe3W, kSe3W, 0, kSe3W);
      bseg(j, P_SE3_B(SE3_W_HID), 0, kSe3W);
      bseg(j, P_SE3_B(SE3_V_HID), kSe3W, kSe3W);
    }
    {
      WgradJob& j = job(s.d_wshead, 16, s.x_se_wv, 2 * kSe3W, 0, 0);
      flush(j, P_SE3_W(SE3_W_OUT), 0, kSe3W, 0, 3, 0, kSe3W);
      flush(j, P_SE3_W(SE3_V_OUT), 0, kSe3W, 3, 3, kSe3W, kSe3W);
      bseg(j, P_SE3_B(SE3_W_OUT), 0, 3);
      bseg(j, P_SE3_B(SE3_V_OUT), 3, 3);
    }
  } else if (!m.nowarp) {
    // warp / sheet layer 0
    {
      WgradJob& j = job(s.d_ws[0], kWarpW, s.x_in_ws, m.KW, 0, 0);
      flush(j, P_WARP_W(0), 0, m.in_w, 0, kWarpW, 0, m.in_w);
      bseg(j, P_WARP_B(0), 0, kWarpW);
      keep(j);
      WgradJob& k = job(s.d_ws[0] + kWarpW / 8, kSheetW, s.x_in_ws, m.KW, 0, 0);
      flush(k, P_SHEET_W(0), 0, m.in_s, 0, kSheetW, 0, m.pe_s);
      flush(k, P_SHEET_W(0), m.pe_s, m.in_s, 0, kSheetW, m.pe_w, m.G);
      bseg(k, P_SHEET_B(0), 0, kSheetW);
      keep(k);
    }
    for (int l = 1; l < kWsDepth; ++l) {
      bool skip = (l == kSkip + 1);
      WgradJob& j = job(s.d_ws[l], kWarpW, s.x_hws[l - 1], kWarpW, s.x_in_ws, skip ? m.KW : 0);
      flush(j, P_WARP_W(l), 0, skip ? ldw5 : kWarpW, 0, kWarpW, 0, skip ? ldw5 : kWarpW);
      bseg(j, P_WARP_B(l), 0, kWarpW);
      keep(j);
      WgradJob& k = job(s.d_ws[l] + kWarpW / 8, kSheetW, s.x_hws[l - 1] + kWarpW / 8, kSheetW, s.x_in_ws, skip ? m.KW : 0);
      if (!skip) {
        flush(k, P_SHEET_W(l), 0, kSheetW, 0, kSheetW, 0, kSheetW);
      } else {
        flush(k, P_SHEET_W(l), 0, lds5, 0, kSheetW, 0, kSheetW + m.pe_s);
        flush(k, P_SHEET_W(l), kSheetW + m.pe_s, lds5, 0, kSheetW, kSheetW + m.pe_w, m.G);
      }
      bseg(k, P_SHEET_B(l), 0, kSheetW);
      keep(k);
    }
    {
      WgradJob& j = job(s.d_wshead, 16, s.x_hws[kWsDepth - 1], kWsW, 0, 0);
      flush(j, P_WARP_W(kWsDepth), 0, kWarpW, 0, 3, 0, kWarpW);
      flush(j, P_SHEET_W(kWsDepth), 0, kSheetW, 3, m.H, kWarpW, kSheetW);
      bseg(j, P_WARP_B(kWsDepth), 0, 3);
      bseg(j, P_SHEET_B(kWsDepth), 3, m.H);
      keep(j);
    }
  }
  const int first_trunk_job = w.njobs;
  // trunk
  {
    WgradJob& j = job(s.d_t[0], kTrunkW, s.x_in_t, m.KT, 0, 0);
    flush(j, P_TRUNK_W(level, 0), 0, m.in_t, 0, kTrunkW, 0, m.in_t);
    bseg(j, P_TRUNK_B(level, 0), 0, kTrunkW);
  }
  for (int l = 1; l <= kTrunkDepth; ++l) {
    bool skip = (l == kSkip + 1);
    int ld = skip ? kTrunkW + m.in_t : kTrunkW;
    WgradJob& j = job(s.d_t[l], kTrunkW, s.x_t[l - 1], kTrunkW, 0, 0);
    flush(j, P_TRUNK_W(level, l), 0, ld, 0, kTrunkW, 0, kTrunkW);
    bseg(j, P_TRUNK_B(level, l), 0, kTrunkW);
    if (skip) {
      WgradJob& k = job(s.d_t[l], kTrunkW, s.x_in_t, m.KT, 0, 0);
      flush(k, P_TRUNK_W(level, l), kTrunkW, ld, 0, kTrunkW, 0, m.in_t);
    }
  }
  {
    WgradJob& j = job(s.d_bott, kRgbW, s.x_t[kTrunkDepth], kTrunkW, 0, 0);
    flush(j, P_BOTT_W(level), 0, kTrunkW, 0, kRgbW, 0, kTrunkW);
    bseg(j, P_BOTT_B(level), 0, kRgbW);
  }
  {
    WgradJob& j = job(s.d_rgb0a, m.n_rgb0a, s.x_bott, kRgbW, s.x_in_v, m.KV);
    flush(j, P_RGB_W(level, 0), 0, ld_rgb0, 0, kRgbW, 0, kRgbW + m.pe_v);
    if (m.cond_r) flush(j, P_RGB_W(level, 0), kRgbW + m.pe_v, ld_rgb0, 0, kRgbW, k_cond, m.G);
    flush(j, P_ALPHA_W(level), 0, ld_alpha, kRgbW, 1, 0, kRgbW);
    if (m.cond_a) flush(j, P_ALPHA_W(level), kRgbW, ld_alpha, kRgbW, 1, k_cond, m.G);
    bseg(j, P_RGB_B(level, 0), 0, kRgbW);
    bseg(j, P_ALPHA_B(level), kRgbW, 1);
  }
  for (int l = 1; l < kRgbDepth; ++l) {
    WgradJob& j = job(s.d_r[l], kRgbW, s.x_r[l - 1], kRgbW, 0, 0);
    flush(j, P_RGB_W(level, l), 0, kRgbW, 0, kRgbW, 0, kRgbW);
    bseg(j, P_RGB_B(level, l), 0, kRgbW);
  }
  {
    WgradJob& j = job(s.d_rgbhead, 16, s.x_r[kRgbDepth - 1], kRgbW, 0, 0);
    flush(j, P_RGB_W(level, kRgbDepth), 0, kRgbW, 0, 3, 0, kRgbW);
    bseg(j, P_RGB_B(level, kRgbDepth), 0, 3);
  }
  // trunk-only job table: everything after the warp / sheet jobs
  WgradTable& wt = plan->wgrad_trunk;
  memset(&wt, 0, sizeof(wt));
  for (int i = first_trunk_job; i < w.njobs; ++i) wt.jobs[wt.njobs++] = w.jobs[i];
  // warp-stage-only job table: the warp / sheet jobs (their slabs lie inside the warp-only stash prefixes)
  WgradTable& ww = plan->wgrad_warp;
  memset(&ww, 0, sizeof(ww));
  for (int i = 0; i < first_trunk_job; ++i) ww.jobs[ww.njobs++] = w.jobs[i];
  (void)d;
}


// ======================================================================================================================
// static baseline: models/nerf.py:41-123 (NeRF(D=8, W=256, in_channels_xyz=63, in_channels_dir=27, skips=[4]))
// ======================================================================================================================
namespace {
struct StaticSlabs {
  uint16_t x_in_x, x_t[kStaticDepth], x_final, x_in_v, x_dir, x_total;
  uint16_t d_t[kStaticDepth], d_final, d_dir, d_rgbhead, d_sigma, d_total;
  uint16_t g_t[kStaticDepth], g_dir, g_total;
  int KX, KV, pe_x, pe_v;
};
StaticSlabs make_static_slabs(const hn_model_desc& d) {
  StaticSlabs s{};
  s.pe_x = 3 + 6 * d.xyz_freqs; s.pe_v = 3 + 6 * d.view_freqs;
  s.KX = pad16(s.pe_x); s.KV = pad16(s.pe_v);
  uint16_t c = 0;
  s.x_in_x = c; c += s.KX / 8;
  for (int l = 0; l < kStaticDepth; ++l) { s.x_t[l] = c; c += kTrunkW / 8; }
  s.x_final = c; c += kTrunkW / 8;
  s.x_in_v = c; c += s.KV / 8;
  s.x_dir = c; c += kRgbW / 8;
  s.x_total = c;
  c = 0;
  for (int l = 0; l < kStaticDepth; ++l) { s.d_t[l] = c; c += kTrunkW / 8; }
  s.d_final = c; c += kTrunkW / 8;
  s.d_dir = c; c += kRgbW / 8;
  s.d_rgbhead = c; c += 2;
  s.d_sigma = c; c += 2;
  s.d_total = c;
  c = 0;
  for (int l = 0; l < kStaticDepth; ++l) { s.g_t[l] = c; c += kTrunkW / 32; }
  s.g_dir = c; c += kRgbW / 32;
  s.g_total = c;
  return s;
}
int static_bias_floats() { return kStaticDepth * kTrunkW + 16 + kTrunkW + kRgbW + 16; }
}  // namespace

static void build_plan_static(const hn_model_desc& d, ModelPlan* plan) {
  const StaticSlabs s = make_static_slabs(d);
  // ---------------------------------------------------------------- forward (nerf.py:84-123)
  {
    Builder b{&plan->fwd, &plan->fwd_logical};
    {   // same rule as make_dims / Shape<>::INB_CHUNKS in hn_mlp.cu
      const int mx = s.KX > s.KV ? s.KX : s.KV;
      const bool in_pad = ones_fit_in_pad(mx, s.KX, s.pe_x) && ones_fit_in_pad(mx, s.KV, s.pe_v);
      b.ones_col = (in_pad ? mx / 8 : mx / 8 + 2) * 8 - 16;
    }
    int bias = 0;
    b.begin_layer(FE_RELU, kTrunkW, bias, s.x_t[0], kNone, s.g_t[0]);
    b.add_op(kTrunkW, s.KX, SRC_INB, 0, 0, SRC_ACT, 0, 0);
    bias += kTrunkW;
    for (int l = 1; l < kStaticDepth; ++l) {
      b.begin_layer(FE_RELU, kTrunkW, bias, s.x_t[l], kNone, s.g_t[l]);
      // skip: cat([input_xyz, h]) (nerf.py:104-106); the hidden part comes first in OUR K order, the packer remaps
      b.add_op(kTrunkW, kTrunkW, SRC_ACT, 0, l == kStaticSkip ? s.KX : 0, SRC_INB, 0, 0);
      bias += kTrunkW;
    }
    b.begin_layer(FE_SIGMA, 16, bias, kNone, kNone);          // sigma = Linear(W, 1)(h8)        nerf.py:109
    b.add_op(16, kTrunkW, SRC_ACT, 0, 0, SRC_ACT, 0, 0);
    bias += 16;
    b.begin_layer(FE_BOTT, kTrunkW, bias, s.x_final, kNone);  // xyz_encoding_final, no activation nerf.py:113
    b.add_op(kTrunkW, kTrunkW, SRC_ACT, 0, 0, SRC_ACT, 0, 0);
    bias += kTrunkW;
    b.begin_layer(FE_RELU, kRgbW, bias, s.x_dir, kNone, s.g_dir);   // dir_encoding on cat([final, dir PE]) nerf.py:115-116
    b.add_op(kRgbW, kTrunkW, SRC_ACT, 0, s.KV, SRC_INB, 0, 0);
    bias += kRgbW;
    b.begin_layer(FE_RGBHEAD, 16, bias, kNone, kNone);        // rgb = Sigmoid(Linear(W/2, 3))   nerf.py:117
    b.add_op(16, kRgbW, SRC_ACT, 0, 0, SRC_ACT, 0, 0);
    bias += 16;
    plan->layout.fwd_off = 0;
    plan->layout.bwd_off = (int64_t)b.w16 * 16;
    without_bias_steps(plan->fwd, &plan->fwd_train);
  }
  // ---------------------------------------------------------------- backward-data
  {
    Builder b{&plan->bwd, &plan->bwd_logical};
    b.begin_layer(BE_MASK, kRgbW, 0, s.d_dir, s.x_dir, s.g_dir);           // rgb^T, A = dY_rgbhead (prologue)
    b.add_op(kRgbW, 16, SRC_ACT, 0, 0, SRC_ACT, 0, 0);
    b.begin_layer(BE_LINEAR, kTrunkW, 0, s.d_final, kNone);                // dir_encoding^T (hidden part)
    b.add_op(kTrunkW, kRgbW, SRC_ACT, 0, 0, SRC_ACT, 0, 0);
    b.begin_layer(BE_MASK, kTrunkW, 0, s.d_t[kStaticDepth - 1], s.x_t[kStaticDepth - 1], s.g_t[kStaticDepth - 1]);
    b.add_op(kTrunkW, kTrunkW, SRC_ACT, 0, 0, SRC_ACT, 0, 0);              // final^T
    b.add_op(kTrunkW, 16, SRC_INB, 0, 0, SRC_ACT, 0, 0, /*acc_init=*/1);   // + sigma^T, A = dY_sigma (prologue, INB)
    for (int l = kStaticDepth - 1; l >= 1; --l) {
      b.begin_layer(BE_MASK, kTrunkW, 0, s.d_t[l - 1], s.x_t[l - 1], s.g_t[l - 1]);
      b.add_op(kTrunkW, kTrunkW, SRC_ACT, 0, 0, SRC_ACT, 0, 0);
    }
    plan->layout.bias_off = plan->layout.bwd_off + (int64_t)b.w16 * 16;
  }
  plan->layout.glo_off = (plan->layout.bias_off + (int64_t)static_bias_floats() * 4 + 15) / 16 * 16;
  plan->layout.total = (plan->layout.glo_off + 255) / 256 * 256;
  PlanInfo& I = plan->info;
  I.x_total = s.x_total; I.d_total = s.d_total; I.g_total = s.g_total;
  I.x_in0 = s.x_in_x; I.x_in_t = kNone; I.x_in_v = s.x_in_v;
  I.d_rgbhead = s.d_rgbhead; I.d_sigma = s.d_sigma;
  I.n_params = HN_NUM_STATIC_PARAM_TENSORS; I.glo_floats = 0; I.glo_param = -1;
  // the descriptor is needed again by build_tables_static: keep the derived sizes in dims (unused otherwise)
  plan->dims.KW = s.KX; plan->dims.KV = s.KV; plan->dims.pe_x = s.pe_x; plan->dims.pe_v = s.pe_v;
}

static void build_tables_static(const int64_t* off, ModelPlan* plan) {
  hn_model_desc d{};
  d.xyz_freqs = (plan->dims.pe_x - 3) / 6; d.view_freqs = (plan->dims.pe_v - 3) / 6;
  const StaticSlabs s = make_static_slabs(d);
  const int pe_x = s.pe_x, pe_v = s.pe_v;
  const int ld_skip = kTrunkW + pe_x, ld_dir = kTrunkW + pe_v;
  PackTable& t = plan->pack;
  memset(&t, 0, sizeof(t));
  Packer pk{&t, off};
  const LogicalOps& F = plan->fwd_logical;
  int oi = 0;
  pk.op(F.ops[oi++]);
  pk.block(SP_TRUNK_W(0), 0, pe_x, 1, 0, kTrunkW, 0, pe_x);
  pk.bias_rows(SP_TRUNK_B(0), 0, kTrunkW);
  for (int l = 1; l < kStaticDepth; ++l) {
    pk.op(F.ops[oi++]);
    if (l == kStaticSkip) {   // weight columns: [0, pe_x) input_xyz, [pe_x, pe_x + W) hidden
      pk.block(SP_TRUNK_W(l), pe_x, ld_skip, 1, 0, kTrunkW, 0, kTrunkW);
      pk.block(SP_TRUNK_W(l), 0, ld_skip, 1, 0, kTrunkW, kTrunkW, pe_x);
    } else {
      pk.block(SP_TRUNK_W(l), 0, kTrunkW, 1, 0, kTrunkW, 0, kTrunkW);
    }
    pk.bias_rows(SP_TRUNK_B(l), 0, kTrunkW);
  }
  pk.op(F.ops[oi++]);
  pk.block(SP_SIGMA_W, 0, kTrunkW, 1, 0, 1, 0, kTrunkW);
  pk.bias_rows(SP_SIGMA_B, 0, 1);
  pk.op(F.ops[oi++]);
  pk.block(SP_FINAL_W, 0, kTrunkW, 1, 0, kTrunkW, 0, kTrunkW);
  pk.bias_rows(SP_FINAL_B, 0, kTrunkW);
  pk.op(F.ops[oi++]);
  pk.block(SP_DIR_W, 0, ld_dir, 1, 0, kRgbW, 0, ld_dir);
  pk.bias_rows(SP_DIR_B, 0, kRgbW);
  pk.op(F.ops[oi++]);
  pk.block(SP_RGB_W, 0, kRgbW, 1, 0, 3, 0, kRgbW);
  pk.bias_rows(SP_RGB_B, 0, 3);

  // backward: dest(n = input feature, k = output feature) = W[k][n]
  const LogicalOps& Bp = plan->bwd_logical;
  const uint32_t bwd16 = (uint32_t)(plan->layout.bwd_off / 16);
  oi = 0;
  auto bop = [&](void) { LogicalOp o = Bp.ops[oi++]; o.w_off16 += bwd16; pk.op(o); };
  bop();  // rgb^T
  pk.block(SP_RGB_W, 0, 1, kRgbW, 0, kRgbW, 0, 3);
  bop();  // dir^T, hidden columns
  pk.block(SP_DIR_W, 0, 1, ld_dir, 0, kTrunkW, 0, kRgbW);
  bop();  // final^T
  pk.block(SP_FINAL_W, 0, 1, kTrunkW, 0, kTrunkW, 0, kTrunkW);
  bop();  // sigma^T
  pk.block(SP_SIGMA_W, 0, 1, kTrunkW, 0, kTrunkW, 0, 1);
  for (int l = kStaticDepth - 1; l >= 1; --l) {
    bop();
    if (l == kStaticSkip) pk.block(SP_TRUNK_W(l), pe_x, 1, ld_skip, 0, kTrunkW, 0, kTrunkW);
    else pk.block(SP_TRUNK_W(l), 0, 1, kTrunkW, 0, kTrunkW, 0, kTrunkW);
  }
  // biases, forward layer order
  int bo = 0;
  for (int l = 0; l < kStaticDepth; ++l) { pk.bias(SP_TRUNK_B(l), bo, kTrunkW); bo += kTrunkW; }
  pk.bias(SP_SIGMA_B, bo, 1); bo += 16;
  pk.bias(SP_FINAL_B, bo, kTrunkW); bo += kTrunkW;
  pk.bias(SP_DIR_B, bo, kRgbW); bo += kRgbW;
  pk.bias(SP_RGB_B, bo, 3); bo += 16;
  t.bias_floats = bo;

  // weight-gradient jobs
  WgradTable& w = plan->wgrad;
  memset(&w, 0, sizeof(w));
  auto job = [&](int dy_chunk, int dy_cols, int x0_chunk, int x0_cols) -> WgradJob& {
    WgradJob& j = w.jobs[w.njobs++];
    j.dy_chunk = (uint16_t)dy_chunk; j.dy_nchunks = (uint16_t)(dy_cols / 8);
    j.x0_chunk = (uint16_t)x0_chunk; j.x0_nchunks = (uint16_t)(x0_cols / 8);
    j.x1_chunk = 0; j.x1_nchunks = 0;
    j.mblocks = (uint8_t)((dy_cols + 127) / 128);
    return j;
  };
  auto flush = [&](WgradJob& j, int param, int64_t extra, int ld, int row0, int nrows, int col0, int ncols) {
    FlushSeg& f = j.flush[j.nflush++];
    f.dst = off[param] + extra; f.ld = ld; f.row0 = (uint16_t)row0; f.nrows = (uint16_t)nrows;
    f.col0 = (uint16_t)col0; f.ncols = (uint16_t)ncols;
  };
  auto bseg = [&](WgradJob& j, int param, int col0, int ncols) {
    BiasSeg& b = j.bias[j.nbias++];
    b.dst = off[param]; b.col0 = (uint16_t)col0; b.ncols = (uint16_t)ncols; b.pad = 0;
  };
  {
    WgradJob& j = job(s.d_t[0], kTrunkW, s.x_in_x, s.KX);
    flush(j, SP_TRUNK_W(0), 0, pe_x, 0, kTrunkW, 0, pe_x);
    bseg(j, SP_TRUNK_B(0), 0, kTrunkW);
  }
  for (int l = 1; l < kStaticDepth; ++l) {
    const bool skip = l == kStaticSkip;
    WgradJob& j = job(s.d_t[l], kTrunkW, s.x_t[l - 1], kTrunkW);
    flush(j, SP_TRUNK_W(l), skip ? pe_x : 0, skip ? ld_skip : kTrunkW, 0, kTrunkW, 0, kTrunkW);
    bseg(j, SP_TRUNK_B(l), 0, kTrunkW);
    if (skip) {
      WgradJob& k = job(s.d_t[l], kTrunkW, s.x_in_x, s.KX);
      flush(k, SP_TRUNK_W(l), 0, ld_skip, 0, kTrunkW, 0, pe_x);
    }
  }
  {
    WgradJob& j = job(s.d_sigma, 16, s.x_t[kStaticDepth - 1], kTrunkW);
    flush(j, SP_SIGMA_W, 0, kTrunkW, 0, 1, 0, kTrunkW);
    bseg(j, SP_SIGMA_B, 0, 1);
  }
  {
    WgradJob& j = job(s.d_final, kTrunkW, s.x_t[kStaticDepth - 1], kTrunkW);
    flush(j, SP_FINAL_W, 0, kTrunkW, 0, kTrunkW, 0, kTrunkW);
    bseg(j, SP_FINAL_B, 0, kTrunkW);
  }
  {
    WgradJob& j = job(s.d_dir, kRgbW, s.x_final, kTrunkW);
    flush(j, SP_DIR_W, 0, ld_dir, 0, kRgbW, 0, kTrunkW);
    bseg(j, SP_DIR_B, 0, kRgbW);
    WgradJob& k = job(s.d_dir, kRgbW, s.x_in_v, s.KV);
    flush(k, SP_DIR_W, kTrunkW, ld_dir, 0, kRgbW, 0, pe_v);
  }
  {
    WgradJob& j = job(s.d_rgbhead, 16, s.x_dir, kRgbW);
    flush(j, SP_RGB_W, 0, kRgbW, 0, 3, 0, kRgbW);
    bseg(j, SP_RGB_B, 0, 3);
  }
}

}  // namespace hn
