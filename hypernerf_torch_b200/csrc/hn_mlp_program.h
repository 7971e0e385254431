// Layer programs for the fused HyperNeRF MLP kernels.
//
// The fused forward / backward-data kernels are interpreters of a small table built on the host from
// hn_model_desc: a list of UMMA "ops" (one accumulation group D[128,N] (+)= A[128,K] * W[N,K]^T, the A
// operand taken from up to two shared-memory column ranges so that skip concatenations never materialise)
// grouped into "layers" (ops that share one TMEM epilogue).  The weight-gradient kernel interprets a table
// of "jobs" (dW = dY^T X over 64-row half tiles).  All of it is plain data so it can be passed by value as
// a kernel parameter.
//
// Topology source: hypernerf/modules.py:99-127 (MLP), :220-252 (NerfMLP), :302-337 (HyperSheetMLP),
// hypernerf/warping.py:74-88 (TranslationField), :128-240 (SE3Field), hypernerf/models.py:404-493 (conditioning, template query).
#pragma once
#include <stdint.h>
#include "../../include/hypernerf_b200.h"

namespace hn {

// One CTA per SM owns 256 samples as two 128-row sub-tiles that share every weight stage.  (Two CTAs of 128 samples per
// SM leave room for only a 2 x 8 KB weight ring, which starves the UMMAs: fwd 2.83 -> 4.06 ms, dgrad 2.78 -> 3.92 ms per
// 1 M samples, profiles/README.md.)
constexpr int kTileRows = 128;   // samples per sub-tile (= UMMA M = TMEM lanes)
constexpr int kSubTiles = 2;
// The inference forward is compiled a second time (HN_MLP_FWD_VARIANT, hn_mlp.cu) with TWO epilogue warpgroups per
// sub-tile, each taking half of the accumulator columns of the wide (ReLU / linear) layers.  A drain is latency bound per
// warp (one warp per scheduler issues ~0.2 instructions per clock: TMEM load -> bias -> pack -> st.shared chains); the
// second warpgroup per sub-tile doubles the drain's memory-level parallelism.  The "primary" warpgroup of a sub-tile also
// does the per-row work (positional encodings, heads); the "secondary" one only drains its column share.
#ifdef HN_MLP_FWD_VARIANT
constexpr int kEpiSplit = 2;
#else
constexpr int kEpiSplit = 1;
#endif
constexpr int kMlpThreads = 128 + 128 * kSubTiles * kEpiSplit;   // epilogue warpgroups (kEpiSplit per sub-tile), then the feeder warpgroup: producer + UMMA issuer
constexpr int kCtaRows = kTileRows * kSubTiles;
constexpr int kHalfRows = 64;    // granularity of the saved-activation layout and of the wgrad K step
constexpr int kChunkBytes = kTileRows * 16;      // one 8-column chunk of a 128-row smem operand
constexpr int kHalfChunkBytes = kHalfRows * 16;  // one 8-column chunk of a 64-row global slab
// weight ring: 3 x 16 KB beside the resident activations (6 x 8 KB measured slower)
constexpr int kRingStages = 3;
constexpr int kStageBytes = 16384;
// Bias folding: in the INFERENCE forward (no stash) every layer's bias rides in the UMMAs: one extra K = 16 step
// whose A operand is the last chunk pair of the input buffer INB — its last two columns hold 1.0 — and whose weight rows
// are [0 x 14, bf16(b), bf16(b - bf16(b))] (two bf16 terms carry the fp32 bias to ~2^-17 relative).  The epilogue then
// has no bias staging (global load -> shared, named barrier) and no LDS + FADD per column.  The ones live in the zero
// padding of the widest input vector when it has >= 2 pad columns (cfg 1: trunk input 89 -> 96), otherwise in one extra
// chunk pair.  Measured per 1 M samples: inference 2.03 -> 1.90 ms; the training forward, whose drain is bound by the
// stash stores and hides the bias adds under them, only pays for the extra K steps (2.76 -> 2.89 ms), so it runs the
// same program without the bias steps (ModelPlan::fwd_train) and adds the biases in its epilogue.
constexpr bool ones_fit_in_pad(int kmax, int k, int in) { return k < kmax || in <= kmax - 2; }
constexpr int kMaxOps = 64;
constexpr int kMaxLayers = 28;
constexpr int kMaxJobs = 40;
constexpr uint16_t kNone = 0xFFFF;

constexpr int pad16(int x) { return (x + 15) / 16 * 16; }

// Fixed cfg-1 family widths (models.py:137-141, warping.py:61, modules.py:303).
constexpr int kTrunkW = 256, kTrunkDepth = 8, kRgbW = 128, kRgbDepth = 4;
constexpr int kWarpW = 128, kSheetW = 64, kWsDepth = 6, kWsW = kWarpW + kSheetW, kSkip = 4;
// SE3Field (warping.py:128-272): trunk depth 6 / width 128 / skip 4 on posenc(points, 0, 8) (8 scales x (sin, cos) x 3 = 48
// columns, no identity, no metadata), a 128 -> 128 logit layer without activation, then the w / v heads: one hidden 128 ReLU
// layer each (run as one 256-wide layer) and 3 outputs each (one 16-row head: rows 0..2 = w, 3..5 = v).
constexpr int kSe3W = 128, kSe3Freqs = 8;
// SE3Field + HyperSheetMLP (HyperNeRF's "DS" model, bendy-sheet slicing, H = 2): the two nets share no input column
// (posenc(points, 0, 8) has no identity columns and non-integer octaves), so their common input vector is
// [posenc(points, 0, 8) 48 | posenc_orig(points, 7) 45 | GLO 8] = 101 -> 112 columns.  That is too wide for INB beside
// the trunk input, so it lives in ACT like the wide trunk inputs (FE_SKIPFEED re-fills it for the skip layer); the merged
// warp stage is 192 wide (SE3 trunk 128 | sheet 64) as in the translation configurations.

// View-direction condition vector of the template (hyper model): [posenc_orig(viewdirs, view_freqs <= 6) zero-padded to 40
// columns | GLO condition (8 columns, zero without template conditioning)] = 48 columns, whatever view_freqs is, so that
// the view frequency count and the conditioning flags are run-time values of one kernel instantiation.
constexpr int kViewPeCols = 40, kViewCondCol = 40, kKV = 48, kMaxViewFreqs = 6;
// The trunk input vector (posenc of the warped point + hyper coordinates) lives in the input buffer INB when it is at
// most this wide (hyper_dim <= 2: 89 -> 96 columns); wider ones (hyper_dim 4: 128, 8: 176 columns) would not leave room
// for the weight ring, so they are written into the activation buffer ACT instead — free at that point — and the skip
// layer, which needs the vector a second time, becomes two layers: the hidden part, then (ACT re-filled with the
// recomputed vector by the FE_SKIPFEED epilogue) the input part accumulating on top.
constexpr int kMaxTrunkInInb = 96;
constexpr int max3(int a, int b, int c) { return a > b ? (a > c ? a : c) : (b > c ? b : c); }
// Shared-input-buffer geometry from the padded vector widths (KW = 0: no warp / sheet stage); used by the compile-time
// Shape<> of hn_mlp.cu and by make_dims, which must agree.
constexpr bool trunk_in_act(int KT) { return KT > kMaxTrunkInInb; }
constexpr int inb_max_cols(int KW, int KT, int KV) { return max3(KW, trunk_in_act(KT) ? 0 : KT, KV); }
constexpr bool inb_ones_in_pad(int KW, int in_w, int KT, int in_t, int KV, int in_v) {
  const int mx = inb_max_cols(KW, KT, KV);
  return (KW == 0 || ones_fit_in_pad(mx, KW, in_w)) && (trunk_in_act(KT) || ones_fit_in_pad(mx, KT, in_t)) &&
         ones_fit_in_pad(mx, KV, in_v);
}
constexpr int inb_chunks_of(int KW, int in_w, int KT, int in_t, int KV, int in_v) {
  const int mx = inb_max_cols(KW, KT, KV);
  return !inb_ones_in_pad(KW, in_w, KT, in_t, KV, in_v) ? mx / 8 + 2 : mx / 8;
}

// Derived channel counts for a model descriptor.
struct Dims {
  int G, H;
  bool nowarp, axis, cond_a, cond_r;   // no warp / sheet stage; hyper point = GLO vector; template GLO conditioning
  bool se3;                            // the warp stage is an SE3Field (no GLO input) instead of a TranslationField
  bool ws_act;                         // SE3Field + HyperSheetMLP: the warp-stage input vector lives in ACT (see kSe3W)
  int ws_w;                            // width of the warp-stage hidden layers: 192 (warp 128 | sheet 64) or 128 (SE3 trunk)
  int pe_w, pe_s, in_w, in_s, KW;  // warp / sheet inputs, shared padded input width (KW = 0 without warp)
  int pe_x, pe_h, in_t, KT;        // trunk input
  int pe_v, KV;                    // view-direction condition: pe_v real posenc columns inside the kKV-wide vector
  int n_rgb0a;                     // rgb layer 0 merged with the alpha head (pad16(128 + 1))
  bool t_in_act;                   // trunk input vector lives in ACT (see kMaxTrunkInInb)
  int inb_chunks;                  // chunks of the shared input buffer (+2 when the ones columns do not fit in padding)
  int ones_col;                    // first column of the chunk pair whose last two columns are 1.0 (bias folding)
};
inline Dims make_dims(const hn_model_desc& d) {
  Dims m{};
  m.se3 = (d.flags & HN_FLAG_WARP_SE3) != 0;
  m.nowarp = (d.flags & (HN_FLAG_WARP_TRANSLATION | HN_FLAG_WARP_SE3)) == 0;
  m.axis = (d.flags & HN_FLAG_SLICE_AXIS) != 0;
  m.ws_act = m.se3 && !m.axis;
  m.ws_w = m.se3 && !m.ws_act ? kSe3W : kWsW;
  m.cond_a = (d.flags & HN_FLAG_ALPHA_COND) != 0; m.cond_r = (d.flags & HN_FLAG_RGB_COND) != 0;
  m.G = d.glo_dim; m.H = m.nowarp ? 0 : d.hyper_dim;
  m.pe_w = 3 + 6 * d.warp_freqs; m.pe_s = 3 + 6 * d.sheet_freqs;
  m.in_w = m.pe_w + m.G; m.in_s = m.pe_s + m.G;
  if (m.se3) { m.pe_w = 6 * d.warp_freqs; m.in_w = m.pe_w; if (!m.ws_act) { m.pe_s = 0; m.in_s = 0; } }
  m.KW = m.nowarp ? 0 : pad16(m.ws_act ? m.in_w + m.in_s : m.in_w);
  m.pe_x = 3 + 6 * d.xyz_freqs; m.pe_h = m.H * (1 + 2 * d.hyper_freqs);
  m.in_t = m.pe_x + m.pe_h; m.KT = pad16(m.in_t);
  m.pe_v = 3 + 6 * d.view_freqs; m.KV = kKV;
  m.n_rgb0a = pad16(kRgbW + 1);
  m.t_in_act = trunk_in_act(m.KT);
  m.inb_chunks = inb_chunks_of(m.ws_act ? 0 : m.KW, m.in_w, m.KT, m.in_t, m.KV, m.pe_v);
  m.ones_col = m.inb_chunks * 8 - 16;
  return m;
}

// ---- canonical parameter tensor indices (include/hypernerf_b200.h) -----------------------------------
constexpr int P_GLO = 0;
inline int P_SHEET_W(int l) { return 1 + 2 * l; }   // l = 0..5 hidden, 6 = logit
inline int P_SHEET_B(int l) { return 2 + 2 * l; }
inline int P_WARP_W(int l) { return 15 + 2 * l; }
inline int P_WARP_B(int l) { return 16 + 2 * l; }
inline int P_LEVEL(int level) { return 29 + 32 * level; }
inline int P_TRUNK_W(int level, int l) { return P_LEVEL(level) + 2 * l; }  // l = 0..7, 8 = logit
inline int P_TRUNK_B(int level, int l) { return P_LEVEL(level) + 2 * l + 1; }
inline int P_BOTT_W(int level) { return P_LEVEL(level) + 18; }
inline int P_BOTT_B(int level) { return P_LEVEL(level) + 19; }
inline int P_RGB_W(int level, int l) { return P_LEVEL(level) + 20 + 2 * l; }  // l = 0..3, 4 = logit
inline int P_RGB_B(int level, int l) { return P_LEVEL(level) + 21 + 2 * l; }
inline int P_ALPHA_W(int level) { return P_LEVEL(level) + 30; }
inline int P_ALPHA_B(int level) { return P_LEVEL(level) + 31; }
constexpr int P_COND_GLO = 93;   // nerf_embed.embed.weight: the condition table without warp
// SE3Field: its trunk (linears 0..5, logit_layer) takes the P_WARP_* slots; the heads follow the condition table
enum Se3Head { SE3_W_HID = 0, SE3_W_OUT = 1, SE3_V_HID = 2, SE3_V_OUT = 3 };
inline int P_SE3_W(int h) { return 94 + 2 * h; }
inline int P_SE3_B(int h) { return 95 + 2 * h; }

// ---- saved-activation (forward) and pre-activation-gradient (backward) slab offsets, in 8-col chunks ---
struct SlabMap {
  // forward activations X (inputs of every linear layer)
  uint16_t x_in_ws, x_hws[kWsDepth], x_in_t, x_t[kTrunkDepth + 1], x_bott, x_in_v, x_r[kRgbDepth];
  uint16_t x_se_logit, x_se_wv;   // SE3: output of the trunk's logit layer (input of the w / v hidden layer), that layer's output
  uint16_t x_total;
  // gradients w.r.t. every layer's pre-activation output
  uint16_t d_ws[kWsDepth], d_wshead, d_t[kTrunkDepth + 1], d_bott, d_rgb0a, d_r[kRgbDepth] /* [0] unused */, d_rgbhead;
  uint16_t d_se_logit, d_se_wv;
  uint16_t d_sheethead;   // SE3 + sheet: the sheet logit layer's dY (16 columns), right after d_wshead
  uint16_t d_total;
  // ReLU gate words (one uint32 per row per 32 output columns of every ReLU layer), written by the forward epilogue
  // next to the X slabs and read by the data gradient instead of the activations themselves
  uint16_t g_hws[kWsDepth], g_t[kTrunkDepth + 1], g_r[kRgbDepth];
  uint16_t g_se_wv;
  uint16_t g_total;
};
inline SlabMap make_slabs(const Dims& m) {
  SlabMap s{};
  uint16_t c = 0;
  s.x_in_ws = c; c += m.KW / 8;
  if (!m.nowarp) for (int l = 0; l < kWsDepth; ++l) { s.x_hws[l] = c; c += m.ws_w / 8; }
  if (m.se3) { s.x_se_logit = c; c += kSe3W / 8; s.x_se_wv = c; c += 2 * kSe3W / 8; }
  s.x_in_t = c; c += m.KT / 8;
  for (int l = 0; l <= kTrunkDepth; ++l) { s.x_t[l] = c; c += kTrunkW / 8; }
  s.x_bott = c; c += kRgbW / 8;
  s.x_in_v = c; c += m.KV / 8;
  for (int l = 0; l < kRgbDepth; ++l) { s.x_r[l] = c; c += kRgbW / 8; }
  s.x_total = c;
  c = 0;
  if (!m.nowarp) {
    for (int l = 0; l < kWsDepth; ++l) { s.d_ws[l] = c; c += m.ws_w / 8; }
    if (m.se3) { s.d_se_logit = c; c += kSe3W / 8; s.d_se_wv = c; c += 2 * kSe3W / 8; }
    s.d_wshead = c; c += 2;
    if (m.ws_act) { s.d_sheethead = c; c += 2; }
  }
  for (int l = 0; l <= kTrunkDepth; ++l) { s.d_t[l] = c; c += kTrunkW / 8; }
  s.d_bott = c; c += kRgbW / 8;
  s.d_rgb0a = c; c += m.n_rgb0a / 8;
  s.d_r[0] = kNone;
  for (int l = 1; l < kRgbDepth; ++l) { s.d_r[l] = c; c += kRgbW / 8; }
  s.d_rgbhead = c; c += 2;
  s.d_total = c;
  c = 0;
  if (!m.nowarp) for (int l = 0; l < kWsDepth; ++l) { s.g_hws[l] = c; c += m.ws_w / 32; }
  if (m.se3) { s.g_se_wv = c; c += 2 * kSe3W / 32; }
  for (int l = 0; l <= kTrunkDepth; ++l) { s.g_t[l] = c; c += kTrunkW / 32; }
  for (int l = 0; l < kRgbDepth; ++l) { s.g_r[l] = c; c += kRgbW / 32; }
  s.g_total = c;
  return s;
}

// ---- fused kernel program ----------------------------------------------------------------------------
enum Src : uint8_t { SRC_ACT = 0, SRC_INB = 1 };

struct MmaOp {
  uint32_t w_off16;            // weights of this op inside the packed blob, 16-byte units
  uint16_t n;                  // UMMA N (multiple of 16)
  uint16_t k;                  // K columns (multiple of 16), all taken from one source buffer
  uint16_t a_chunk;            // first 8-col chunk inside the source buffer
  uint16_t tmem_col;           // accumulator column offset
  uint8_t src;
  uint8_t acc_init;            // 1: accumulate onto what TMEM already holds
  uint8_t cps;                 // 8-col chunks of K per ring stage (even)
  uint8_t pad;                 // 1: bias K step (bias folding), dropped from ModelPlan::fwd_train
  uint16_t kc0, kc_total;      // first chunk of this op inside its logical weight matrix / that matrix's chunk count
};
// A weight matrix as the packer sees it: one [n x k] operand image; a skip layer's matrix is consumed by two
// consecutive MmaOps (hidden part, then input part accumulating on top).
struct LogicalOp {
  uint32_t w_off16;
  uint16_t n, k;
};

// FE_SKIPFEED: no drain — the accumulator keeps the hidden part of the skip layer; the epilogue re-fills ACT with the trunk
// input vector for the input part (see kMaxTrunkInInb).  BE_LINCOND: BE_LINEAR + the GLO-condition columns (-> table gradient).
// FE_LINEAR: plain linear layer (bias, no activation, stashed): the SE3 trunk's logit layer.
// SE3 + sheet (Dims::ws_act): FE_SKIPFEED re-fills ACT[0, KW) with the warp-stage input vector instead; FE_LINSHEET is
// FE_LINEAR on the SE3 logit columns [0, 128) plus the sheet's logit layer (64 -> H) in columns [128, 144), whose H hyper
// coordinates the epilogue keeps for FE_WSHEAD (the next layer's 256-wide output overwrites all of ACT).  BE_LINSHEET is
// BE_LINEAR plus the sheet head's dY (kept since BE_TRUNKIN) written to ACT[128, 144) for the (SE3 logit | sheet logit)^T layer.
// Tangent program (ModelPlan::fwd_warp_tangent, PF_TANGENT): FE_TANGENT replaces FE_RELU — no bias, the bf16 output masked
// with the PRIMAL sample's gate words of the layer (Layer::gate_word is read, not written); FE_JACHEAD replaces FE_WSHEAD
// and writes jac[n, r, c] = acc[r] + (r == c), r < 3, for the launch's input direction c.
enum FwdEpi : uint8_t { FE_RELU = 0, FE_WSHEAD, FE_BOTT, FE_RGB0A, FE_RGBHEAD, FE_SIGMA, FE_SKIPFEED, FE_LINEAR, FE_LINSHEET,
                        FE_TANGENT, FE_JACHEAD };
enum BwdEpi : uint8_t { BE_MASK = 0, BE_LINEAR, BE_RGB1, BE_SKIPSTORE, BE_TRUNKIN, BE_GLO, BE_LINCOND, BE_LINSHEET };
// PF_WARP_ONLY: a warp-stage-only program (ModelPlan::fwd_warp*, bwd_warp).  Its forward ends at the FE_WSHEAD epilogue,
// which then writes `warped` (and the SE3 screw) but no trunk input; its data gradient starts at the head^T layer, whose
// A operand the prologue builds from the upstream g_warped instead of from the rgb head.
// PF_TANGENT: the bias-free gated linear pass of the translation warp stage along one input direction (hn_mlp_fwd_warp_tangent).
enum ProgFlags : int32_t { PF_TIN_ACT = 1, PF_WARP_ONLY = 2, PF_TANGENT = 4 };   // Program::flags

struct Layer {
  uint8_t op0, nops, epi, pad;
  uint16_t n_out;       // accumulator columns the epilogue consumes
  uint16_t bias_off;    // forward: float offset into the bias array
  uint16_t save_chunk;  // chunk offset where the epilogue's bf16 output is stashed (X slabs fwd, dY slabs bwd)
  uint16_t mask_chunk;  // backward: chunk offset of the forward activation that gates this gradient (kNone: no gate)
  uint16_t gate_word;   // first ReLU gate word of this layer's output (forward: written, backward: read); kNone: none
  uint16_t pad2;
};

struct Program {
  int32_t nlayers, nops;
  int32_t flags, pad;
  Layer layers[kMaxLayers];
  MmaOp ops[kMaxOps];
};
struct LogicalOps {
  int32_t n;
  LogicalOp ops[kMaxOps];
};

// ---- weight packing ----------------------------------------------------------------------------------
// dest(n, k) of an op's [N x K] bf16 matrix (interleave layout: ((k/8) * N + n) * 8 + k%8) is gathered from
// flat_params[src + (n - n0) * sn + (k - k0) * sk] for the (n, k) inside a block; everything else is zero.
constexpr int32_t kBiasPairStride = INT32_MIN;   // PackBlock::sk marker: rows k0, k0 + 1 = bf16(b[n]), bf16(b[n] - bf16(b[n]))
// Positional-encoding window (include/hypernerf_b200.h, hn_pack_weights_windowed): a block / flush segment whose source
// columns are encoded columns of one encoder carries the encoder's window spec.  The source column runs along k for the
// forward images (sk == 1) and along n for the transposed ones (sn == 1); for a weight-gradient segment along its columns.
// Encoded column e = win_e0 + (offset along that axis); with identity columns first (kWinIdentity), e < C is identity.
// win = 1 + the index of the encoder's alpha in pe_alpha, 0 (kNoWin, what a zeroed table holds) for none.
enum PeAlpha : uint8_t { PE_WARP = 0, PE_SHEET = 1, PE_NERF = 2, PE_HYPER = 3, kNumPeAlphas = 4 };
constexpr uint8_t kNoWin = 0;
constexpr uint8_t kWinIdentity = 0x80;  // win_c flag: C identity columns precede the bands; low 7 bits = C
struct PackBlock {
  int64_t src;         // element offset in the flat fp32 parameter buffer
  int32_t sn, sk;      // source strides (elements)
  uint16_t n0, nn, k0, kk;
  uint8_t win, win_c;  // window: 1 + pe_alpha index (kNoWin: none), channels | kWinIdentity
  uint16_t win_e0;     // encoded column of the block's first source column
};
struct PackOp {
  uint32_t w_off16;
  uint16_t n, k;       // padded dims
  uint8_t blk0, nblk;
  uint16_t pad;
};
constexpr int kMaxPackOps = 64;
constexpr int kMaxPackBlocks = 160;
struct BiasBlock { int64_t src; uint16_t dst, cnt; uint32_t pad; };
constexpr int kMaxBiasBlocks = 40;
struct PackTable {
  int32_t nops, nblocks, nbias, bias_floats;
  PackOp ops[kMaxPackOps];
  PackBlock blocks[kMaxPackBlocks];
  BiasBlock bias[kMaxBiasBlocks];
};

// ---- weight-gradient jobs ----------------------------------------------------------------------------
struct FlushSeg {
  int64_t dst;           // element offset in flat_grad of D[row0][col0]
  int32_t ld;            // destination leading dimension
  uint16_t row0, nrows;  // rows in dY-column space of the job (row = mblock * 128 + lane row)
  uint16_t col0, ncols;
  uint8_t win, win_c;    // window of the columns (PackBlock): the flush scales dY^T pe by w
  uint16_t win_e0;
};
struct BiasSeg { int64_t dst; uint16_t col0, ncols; uint32_t pad; };
struct WgradJob {
  uint16_t dy_chunk, dy_nchunks;   // dY columns copied as the A operand
  uint16_t x0_chunk, x0_nchunks;   // X columns (first range) copied as the B operand
  uint16_t x1_chunk, x1_nchunks;   // optional second range, placed right after the first
  uint8_t mblocks;                 // 1 or 2 blocks of 128 dY columns
  uint8_t nflush, nbias, group;    // group: which CTA group owns this job (hn_mlp.cu: kWgGroups)
  FlushSeg flush[4];
  BiasSeg bias[2];
};
struct WgradTable {
  int32_t njobs;
  int32_t pad;
  WgradJob jobs[kMaxJobs];
};

// Layout of one level's packed blob.
struct PackedLayout {
  int64_t fwd_off, bwd_off, bias_off, glo_off, total;  // bytes
};

// What the host launch code needs to know about a plan, whichever model family built it.
struct PlanInfo {
  uint16_t x_total, d_total, g_total;   // chunks per half tile of the X / dY stashes, gate words per row
  uint16_t x_in0, x_in_t, x_in_v;       // X slabs written by the prologue / trunk-input / view-direction PE
  uint16_t d_rgbhead, d_sigma;          // dY slabs written by the data-gradient prologue
  // Warp-stage-only stash (ModelPlan::fwd_warp*): the X slabs, dY slabs and gate words of the warp / sheet stage are
  // prefixes of their maps (make_slabs), so their prefix lengths serve as the per-half-tile strides; 0 without warp
  uint16_t x_warp, d_warp, g_warp;
  int32_t n_params;                     // canonical parameter tensors
  int32_t glo_floats;
  int32_t glo_param;                    // canonical index of the GLO table the kernels read (copied into the blob); -1: none
};

// static baseline (models/nerf.py): canonical parameter indices = state_dict order
inline int SP_TRUNK_W(int l) { return 2 * l; }   // l = 0..7: xyz_encoding_{l+1}.0
inline int SP_TRUNK_B(int l) { return 2 * l + 1; }
constexpr int SP_FINAL_W = 16, SP_FINAL_B = 17, SP_DIR_W = 18, SP_DIR_B = 19, SP_SIGMA_W = 20, SP_SIGMA_B = 21,
              SP_RGB_W = 22, SP_RGB_B = 23;
constexpr int kStaticDepth = 8, kStaticSkip = 4;   // NeRF(D=8, W=256, skips=[4])

struct ModelPlan {
  Dims dims;
  SlabMap slabs;
  PlanInfo info;
  Program fwd, bwd;
  Program fwd_train;  // fwd without the bias K steps: the stash-writing forward adds biases in its epilogue
  // Trunk-only programs (hyper model): the template NeRF (trunk, bottleneck, rgb / alpha heads) for rows whose warped
  // point and hyper coordinates are already known — the fine level inherits the coarse depths, and the warp / sheet nets
  // are shared between the levels, so those rows' warp / sheet evaluations are the coarse pass's (hn_mlp_fwd_trunk).
  Program fwd_trunk, fwd_trunk_train, bwd_trunk;
  WgradTable wgrad_trunk;   // built per call next to `wgrad`
  // Warp-stage-only programs (models with warp): the layers from the input encoding up to and including the FE_WSHEAD
  // head, and their transposes, flagged PF_WARP_ONLY (hn_mlp_fwd_warp / hn_mlp_bwd_warp_*): `apply_warp` and the
  // background loss need `warped` alone, not the template behind it.
  Program fwd_warp, fwd_warp_train, bwd_warp;
  // Translation warp only: fwd_warp_train with FE_TANGENT / FE_JACHEAD epilogues, flagged PF_WARP_ONLY | PF_TANGENT
  // (hn_mlp_fwd_warp_tangent): the columns of the warp's Jacobian, J[:, c] = e_c + W_head D_L W_L ... D_1 W_1 dPE/dx_c.
  Program fwd_warp_tangent;
  WgradTable wgrad_warp;    // built per call next to `wgrad`
  LogicalOps fwd_logical, bwd_logical;
  PackTable pack;     // needs param_offsets -> built per call
  WgradTable wgrad;   // needs param_offsets -> built per call
  PackedLayout layout;
};

inline bool is_static(const hn_model_desc& d) { return (d.flags & HN_FLAG_STATIC_NERF) != 0; }
// Validates the descriptor; returns 0 or a negative error code (message through set_error).
int validate_desc(const hn_model_desc& d);
// Static part (programs, slabs, blob layout).
void build_plan(const hn_model_desc& d, ModelPlan* plan);
// Offset-dependent part for one level.  windowed: blocks / flush segments are split at the encoder boundaries and carry
// window specs (the unwindowed tables are the same as without the feature).
void build_tables(const hn_model_desc& d, int level, const int64_t* param_offsets, bool windowed, ModelPlan* plan);

}  // namespace hn
