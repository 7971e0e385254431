// Fused HyperNeRF MLP stack for sm_100a: tcgen05 UMMA with TMEM accumulators, weights streamed from L2 by
// 1-D bulk async copies through an mbarrier ring, activations resident in shared memory across layers,
// positional encodings computed in-kernel.
//
//   mlp_fwd_kernel    render_samples -> query_template (models.py:587-650, :447-493): GLO lookup, posenc_orig,
//                     TranslationField (or SE3Field: posenc(0, 8), w / v heads, fp32 exp map), HyperSheetMLP (or the
//                     axis-aligned hyper point), NerfMLP, noise_regularize, Softplus / Sigmoid.
//   mlp_dgrad_kernel  the autograd of the above w.r.t. every layer's pre-activation (and the GLO table).
//   mlp_wgrad_kernel  dW = dY^T X and db = sum dY over all samples, accumulated into the flat gradient.
//   pack_kernel       fp32 (out,in) nn.Linear weights -> bf16 operand images (forward and transposed).
//
// One CTA (one per SM) owns 256 samples as two 128-row sub-tiles (128 = UMMA M = TMEM lanes).  Inference forward: both
// sub-tiles consume every weight stage in lock step, so each byte fetched from L2 feeds two UMMAs.  Training forward and
// data gradient: the sub-tiles run out of phase (Sched<PP>), one draining its accumulator and writing its stash while
// the other's UMMAs run.  384 threads = 3 warpgroups: warpgroups 0-1 are the epilogue (thread = sample row, one
// warpgroup per sub-tile, setmaxnreg 216); the last warpgroup holds the weight producer (one thread, 3 x 16 KB bulk-copy
// ring; 5-6 stages in the data gradient) and the UMMA issuer (one elected thread) and gives its registers away.
// TMEM: 512 columns = 2 sub-tiles x 256 fp32 accumulator columns.  Stash stores are streaming (st.global.cs).
#include <math.h>
#include <algorithm>
#include <string.h>
#include <string>
#include <type_traits>
#include <unordered_map>
#include "hn_api_internal.h"
#include "hn_mlp_program.h"
#include "hn_ptx.cuh"

// This file is compiled twice into libhypernerf_b200.so (Makefile).  The second compilation (hn_mlp_fv.o:
// -DHN_MLP_FWD_VARIANT=1) holds the INFERENCE forward kernels with two epilogue warpgroups per sub-tile (hn_mlp_program.h:
// kEpiSplit), in their own namespace, and exports only hn_mlp_fwd_fv / hn_mlp_fwd_trunk_fv / hn_mlp_fwd_warp_fv, which the
// first compilation's hn_mlp_fwd / hn_mlp_fwd_trunk / hn_mlp_fwd_warp call for every launch without a stash.  Measured
// per 1 M samples in isolation: inference forward 2.03 -> 1.93 ms, training forward 2.50 -> 2.42 ms, data gradient +2 %; a full-frame render goes from 2.27 to
// 2.40 Mrays/s, while inside the power-capped training step the split training forward is a wash (690 k against 691 k
// rays/s over three alternating runs, the trunk-only launch 3 % slower), so training keeps the single-warpgroup kernels.
// The stash / gate-word layout does not depend on the epilogue split.
#ifdef HN_MLP_FWD_VARIANT
namespace hn_fv { using namespace hn; }
#define hn hn_fv
#define hn_mlp_fwd hn_mlp_fwd_fv
#define hn_mlp_fwd_trunk hn_mlp_fwd_trunk_fv
#define hn_mlp_fwd_warp hn_mlp_fwd_warp_fv
#define HN_FV_HIDDEN __attribute__((visibility("hidden")))
#else
#define HN_FV_HIDDEN
#endif

namespace hn {

// out-of-range metadata id inside the fused kernels (HN_TRAP_IDS): see hn_check_ids
#ifndef HN_TRAP_IDS
#define HN_TRAP_IDS 1
#endif
#if HN_TRAP_IDS
#define HN_CHECK_ID(id, n) do { if ((uint64_t)(id) >= (uint64_t)(n)) __trap(); } while (0)
#else
#define HN_CHECK_ID(id, n) do { } while (0)
#endif

// ------------------------------------------------------------------------------------------------------
// compile-time model shape (cfg-1 family of BASELINE.json)
// ------------------------------------------------------------------------------------------------------
template <int G_, int H_, int WF_, int SF_, int XF_, int HF_, int VF_, bool STATIC_ = false, bool SE3_ = false>
struct Shape {
  static constexpr bool STATIC = STATIC_;   // static baseline models/nerf.py: no GLO / warp / sheet / hyper coordinates
  static constexpr bool NOWARP = !STATIC_ && H_ == 0;   // NerfModel(use_warp=False): the template alone on the raw points
  static constexpr bool SE3 = SE3_;         // warp stage = SE3Field (warping.py:128-240): input posenc(points, 0, WF) alone
  // SE3Field + HyperSheetMLP (bendy sheet, SF > 0): the 192-wide merged warp stage reads the vector
  // [posenc(points, 0, WF) | posenc_orig(points, SF) | GLO], held in ACT (hn_mlp_program.h: kSe3W)
  static constexpr bool WS_ACT = SE3_ && SF_ > 0;
  static constexpr int G = G_, H = H_, WF = WF_, SF = SF_, XF = XF_, HF = HF_;
  static constexpr int VF = VF_;            // hyper model: the MAXIMUM view frequency count (run time: FwdParams::view_freqs)
  static constexpr int PE_S = 3 + 6 * SF;
  static constexpr int PE_W = SE3 ? 6 * WF : 3 + 6 * WF, IN_W = WS_ACT ? PE_W + PE_S + G : SE3 ? PE_W : PE_W + G,
                       KW = NOWARP ? 0 : pad16(IN_W);
  static constexpr int PE_X = 3 + 6 * XF, PE_H = H * (1 + 2 * HF), IN_T = PE_X + PE_H, KT = pad16(IN_T);
  static constexpr int PE_V = 3 + 6 * VF, KV = STATIC ? pad16(PE_V) : kKV;
  static constexpr bool TIN_ACT = !STATIC && trunk_in_act(KT);   // trunk input vector in ACT (hn_mlp_program.h: kMaxTrunkInInb)
  // bias folding (hn_mlp_program.h): the last two columns of INB's last chunk pair hold 1.0; they sit in
  // the zero padding of the widest input vector when every vector that reaches the last chunk has >= 2 pad columns
  static constexpr int INB_CHUNKS = STATIC ? inb_chunks_of(KW, IN_W, 0, 0, KV, PE_V)
                                           : inb_chunks_of(WS_ACT ? 0 : KW, IN_W, KT, IN_T, KV, PE_V);
  static_assert(!(WS_ACT && TIN_ACT), "one input vector in ACT per model: FE_SKIPFEED serves either the warp stage or the trunk");
  static constexpr int N_RGB0A = pad16(kRgbW + 1);
  static constexpr int NWARPED = 3 + H;     // columns of a warped point + hyper coordinates
};
using Cfg1 = Shape<8, 2, 10, 7, 10, 6, 6>;
using CfgH4 = Shape<8, 4, 10, 7, 10, 6, 6>;   // opt.py default hyper_slice_out_dim (opt.py:92)
using CfgH8 = Shape<8, 8, 10, 7, 10, 6, 6>;   // bendy sheet with 8 outputs, or axis-aligned slicing (hyper point = GLO vector)
using CfgT = Shape<8, 0, 10, 7, 10, 6, 6>;    // no warp: template NeRF on the raw points
using CfgStatic = Shape<0, 0, 10, 0, 10, 0, 4, true>;   // NeRF(): xyz PE 63 (-> K 64), dir PE 27 (-> K 32)
using CfgSE3 = Shape<8, 8, kSe3Freqs, 0, 10, 6, 6, false, true>;   // config 5: SE3 warp + axis-aligned slicing (hyper point = GLO vector)
using CfgSE3S = Shape<8, 2, kSe3Freqs, 7, 10, 6, 6, false, true>;  // SE3 warp + bendy sheet with 2 outputs (HyperNeRF's "DS" model)

// ------------------------------------------------------------------------------------------------------
// shared memory plan of the fused kernels
// ------------------------------------------------------------------------------------------------------
// Ping-pong schedule: the two sub-tiles of a CTA run half a step out of phase: each has its own accumulator /
// activation barriers and makes its own pass over a layer's weight stages, so sub-tile 0's epilogue (TMEM drain,
// stash stores) runs under sub-tile 1's UMMAs and vice versa.  Price: every weight stage is fetched from L2 once per
// 128 instead of once per 256 samples, i.e. the weight ring has to sustain twice the rate over the same ~1 100-cycle
// refill latency.  Lock step: both sub-tiles consume each stage back to back.
// The training forward and the data gradient run out of phase, the inference forward in lock step.  Measured per 1 M
// samples once the stash stores stopped evicting the weights from L2 (streaming stores): data gradient (80 KB ring)
// 2.55 -> 2.31 ms, training forward (48 KB ring) 2.50 -> 2.42 ms out of phase; inference forward (48 KB ring, short
// drains, bias K steps streamed twice) 1.89 -> 2.34 ms, so it stays in lock step.
template <bool PP>
struct Sched {
  static constexpr int CHAINS = PP ? kSubTiles : 1;          // independently synchronised sub-tile groups
  static constexpr int SUBS = kSubTiles / CHAINS;            // sub-tiles per chain
};
// Warp roles.  The epilogue warpgroups come FIRST and the feeder warpgroup (weight producer, UMMA issuer) LAST: the SM's
// warp arbiter favours the highest warp id, and once a drain loop of one sub-tile runs concurrently with the other
// sub-tile's UMMAs low-numbered feeder warps were starved of issue slots.
constexpr int kEpiWarps = 4 * kSubTiles * kEpiSplit;
// Register budgets after setmaxnreg (feeder / primary / secondary warpgroups).  setmaxnreg moves registers inside the CTA's
// LAUNCH allocation only: 384 threads x 168 = 64 512 with one epilogue warpgroup per sub-tile (128 x 72 + 256 x 216;
// 88 / 208 and 104 / 200: no gain), 640 x 96 = 61 440 with the split epilogue (128 x 72 + 256 x 136 + 256 x 64).  The
// weight producer spills below 72 registers (a split build with 40 / 144 / 72 ran the forward in 2.76 ms per 1 M samples).
constexpr int kRegsFeeder = 72;
constexpr int kRegsPrimary = kEpiSplit == 2 ? 136 : 216;
constexpr int kRegsSecondary = 64;
static_assert(kEpiSplit == 2 ? 128 * kRegsFeeder + 256 * kRegsPrimary + 256 * kRegsSecondary <= 640 * 96
                             : 128 * kRegsFeeder + 256 * kRegsPrimary <= 384 * 168, "register budget");
constexpr int kProducerWarp = kEpiWarps, kIssuerWarp = kEpiWarps + 1;

template <int INB_CHUNKS_, int STAGES_>
struct SmemPlan {
  static constexpr int STAGES = STAGES_;
  static constexpr int ACT_BYTES = 32 * kChunkBytes;              // 128 x 256 bf16 per sub-tile
  static constexpr int INB_BYTES = INB_CHUNKS_ * kChunkBytes;     // 128 x (INB_CHUNKS*8) bf16 per sub-tile
  static constexpr int ACT = 0;
  static constexpr int INB = ACT + kSubTiles * ACT_BYTES;
  static constexpr int RING = INB + kSubTiles * INB_BYTES;        // STAGES x kStageBytes
  static constexpr int BIAS = RING + STAGES * kStageBytes;        // 2 x 256 fp32: this / next layer's bias
  static constexpr int BARS = BIAS + 2 * 256 * 4;                 // full[], empty[], acc_full[2], act_ready[2]
  static constexpr int TMEMP = BARS + (2 * STAGES + 4) * 8;
  static constexpr int TOTAL = TMEMP + 16;
  static_assert(TOTAL <= 227 * 1024, "shared memory budget");
};
// forward: INB holds the PE input vectors (UMMA operands of the first / skip / view layers)
template <class C>
using Smem = SmemPlan<C::INB_CHUNKS, kRingStages>;
// backward-data: INB only holds the 16-column head gradient of the static model, so the weight ring gets the space:
// 5 stages, 6 for the hyper model, whose data gradient keeps nothing in INB at all.  With 3 stages of 512 cycles of UMMA
// work a refill (commit -> producer -> L2 -> complete_tx, ~1 100 cycles after the stage's last UMMA retires) lands ~80
// cycles after the issuer needs the slot again: 12 % of the issuer's time was spent waiting for stages.
template <class C>
using SmemBwd = SmemPlan<C::STATIC ? 2 : 0, C::STATIC ? 5 : 6>;

// run-time model flags of the fused kernels (from hn_model_desc::flags)
enum ModelFlags : int { MF_AXIS = 1, MF_COND = 2 };   // hyper point = GLO vector; GLO condition columns in the view vector
static bool has_warp(const hn_model_desc& d) { return (d.flags & (HN_FLAG_WARP_TRANSLATION | HN_FLAG_WARP_SE3)) != 0; }

struct FwdParams {
  Program prog;
  const uint8_t* weights;   // packed blob base + fwd_off
  const float* bias;        // packed blob base + bias_off
  const float* glo;         // (E, G) fp32 copy of the GLO table
  const float* points; const float* viewdirs; const int64_t* ids; const float* noise;
  const float* warped_in;   // trunk-only program (hn_mlp_fwd_trunk): (n, 3 + H) warped points + hyper coordinates, else NULL
  // Scattered rows: launch row j of ray b reads its point / noise and writes its outputs at position pos[b * S + j] of a
  // (B, S_full) row; NULL = the launch rows ARE the output rows (S_full == S).  The stash stays in launch order.
  const int32_t* pos;
  int S_full;
  float noise_std;
  int view_freqs;           // hyper model: posenc_orig frequencies of the view direction (<= kMaxViewFreqs), run time
  int mflags;               // MF_*
  int n_embed;              // rows of the GLO table: an id outside [0, n_embed) traps (nn.Embedding raises, modules.py:155-167)
  int64_t n;                // samples = B * S
  int S;
  int n_tiles;
  int x_total;              // chunks per half tile of the saved-activation slab
  uint16_t x_in_ws, x_in_t, x_in_v;
  float* sigma; float* rgb; float* warped;
  float* aux;               // SE3 warp, training: (n, 6) screw parameters (w, v) of every launch row for the data gradient
  uint8_t* saved;
  uint32_t* gates;          // ReLU gate words: [half tile][g_total][64 rows] (inside `saved`, after the X slabs)
  int g_total;
  unsigned long long* dbg;  // optional per-CTA cycle counters (hn_debug_set_timing_buffer)
  // tangent launch (mlp_fwd_kernel<C, true, true>): (n, 3, 3) Jacobian of the translation warp.  `gates` are then the PRIMAL
  // stash's gate words, `saved` the nullable tangent stash of 3 planes of x_total X chunks + g_total (unwritten) gate words
  // per half tile each, and n_tiles counts 3 x the primal tiles (plane = tile / primal tiles).
  float* jac;
};

struct BwdParams {
  Program prog;
  const uint8_t* weights;   // packed blob base + bwd_off
  const int64_t* ids;
  const float* sigma; const float* rgb; const float* warped;
  const float* g_sigma; const float* g_rgb; const float* g_warped;
  const float* points; const float* aux;   // SE3 warp: the sample points ((B, S_full) rows) and the forward's (w, v) (launch rows)
  float* g_warped_out;      // trunk-only program: (n, 3 + H) gradient w.r.t. warped_in, written by the last layer; else NULL
  const int32_t* pos;       // scattered rows (see FwdParams): sigma / rgb / g_sigma / g_rgb / g_warped (and, outside the
  int S_full;               // trunk-only program, warped) are indexed at pos[b * S + j] of (B, S_full) rows
  const uint8_t* saved;     // forward stash (X slabs; only its gate-word region is read here)
  const uint32_t* gates;    // ReLU gate words written by the forward: [half tile][g_total][64 rows]
  int g_total;
  uint8_t* dsaved;          // pre-activation gradients for the wgrad kernel
  float* glo_grad;          // flat_grad + offset of the GLO table
  int mflags;               // MF_*
  int n_embed;
  int64_t n;
  int S;
  int n_tiles;
  int x_total, d_total;
  uint16_t d_rgbhead, d_sigma;
  unsigned long long* dbg;
};

// ------------------------------------------------------------------------------------------------------
// weight producer and MMA issuer (shared by forward and backward-data kernels)
// ------------------------------------------------------------------------------------------------------
// cycle counters per CTA: [0] producer wait-empty, [1] mma wait-act_ready, [2] mma wait-full, [3] mma total,
// [4] epilogue wait-acc_full, [5] epilogue work, [6] epilogue prologue, [7] epilogue total
#ifndef HN_ROLE_TIMING
#define HN_ROLE_TIMING 0   // make EXTRA=-DHN_ROLE_TIMING=1 for profiles/role_timing.py
#endif
#if HN_ROLE_TIMING
#define HN_T0() (clock64())
#else
#define HN_T0() (0ll)
#endif
template <int STAGES>
struct RingStateT { int slot = 0; uint32_t phase = 0; __device__ void next() { if (++slot == STAGES) { slot = 0; phase ^= 1; } } };
using RingState = RingStateT<kRingStages>;

template <bool PP, class RS>
__device__ __forceinline__ void produce_tile(const Program& prog, const uint8_t* __restrict__ weights, uint8_t* ring,
                                             uint64_t* full, uint64_t* empty, RS& rs, long long& t_wait) {
  for (int li = 0; li < prog.nlayers; ++li) {
    const Layer& L = prog.layers[li];
    for (int chain = 0; chain < Sched<PP>::CHAINS; ++chain) {   // ping-pong: every sub-tile makes its own pass over the layer
      for (int oi = L.op0; oi < L.op0 + L.nops; ++oi) {
        const MmaOp& op = prog.ops[oi];
        const int nchunks = op.k >> 3;
        const uint8_t* src = weights + (size_t)op.w_off16 * 16;
        for (int c = 0; c < nchunks; c += op.cps) {
          int cnt = min((int)op.cps, nchunks - c);
          uint32_t bytes = (uint32_t)cnt * op.n * 16;
          long long t0 = HN_T0();
          mbar_wait(&empty[rs.slot], rs.phase ^ 1);
          t_wait += HN_T0() - t0;
          mbar_arrive_expect_tx(&full[rs.slot], bytes);
          bulk_g2s(ring + rs.slot * kStageBytes, src + (size_t)c * op.n * 16, bytes, &full[rs.slot]);
          rs.next();
        }
      }
    }
  }
}

// The issuing thread's own instruction stream bounds the tensor pipe: measured with profiles/umma_rate{2,3}.py, a
// UMMA retires at its floor (N/2 cycles for N >= 128) only if the issue loop spends less than that per instruction.
// So everything that can be hoisted is: per op the descriptors' low words are formed once, and the k-step loop only
// adds constants to them (address field = bits [0,14) of the low word, in 16-byte units; smem addresses stay below
// 256 KB so the add never carries into the LBO field).
constexpr uint32_t kDescHi = (1u << 14) | (128u >> 4);   // descriptor version 1, SBO = 128 B, no swizzle
__device__ __forceinline__ uint64_t desc64(uint32_t lo) { return ((uint64_t)kDescHi << 32) | lo; }

template <bool PP, class RS>
__device__ __forceinline__ void issue_layer(const Program& prog, const Layer& L, int sub0, uint32_t act_s, uint32_t inb_s,
                                            uint32_t act_stride, uint32_t inb_stride, uint32_t ring_s,
                                            uint32_t tmem_base, uint64_t* full, uint64_t* empty, RS& rs,
                                            long long& t_wait) {
  for (int oi = L.op0; oi < L.op0 + L.nops; ++oi) {
    const MmaOp& op = prog.ops[oi];
    const uint32_t n = op.n, nchunks = op.k >> 3, cps = op.cps;
    const uint32_t idesc = make_idesc_bf16(kTileRows, n, 0, 0);
    const bool from_act = op.src == SRC_ACT;
    // A: K-major, LBO = one 8-column chunk of 128 rows
    const uint32_t a_sub = (from_act ? act_stride : inb_stride) >> 4;
    const uint32_t a_base = ((((from_act ? act_s : inb_s) + op.a_chunk * kChunkBytes) >> 4) | ((uint32_t)(kChunkBytes >> 4) << 16)) + sub0 * a_sub;
    const uint32_t d0 = tmem_base + op.tmem_col + sub0 * 256;
    const uint32_t acc0 = op.acc_init;
    for (uint32_t c = 0; c < nchunks; c += cps) {
      const uint32_t cnt = min(cps, nchunks - c);
      long long t0 = HN_T0();
      mbar_wait(&full[rs.slot], rs.phase);
      t_wait += HN_T0() - t0;
      tc_fence_after();
      if (elect_one_sync()) {
        uint32_t a_lo = a_base + c * (uint32_t)(kChunkBytes >> 4);
        uint32_t b_lo = ((ring_s + rs.slot * kStageBytes) >> 4) | (n << 16);   // B: K-major, LBO = N * 16 B
        uint32_t acc = (c > 0) | acc0;
        for (uint32_t j = 0; j < cnt; j += 2) {
          const uint64_t bd = desc64(b_lo);
#pragma unroll
          for (int sub = 0; sub < Sched<PP>::SUBS; ++sub) umma_bf16(d0 + sub * 256, desc64(a_lo + sub * a_sub), bd, idesc, acc);
          a_lo += 2 * (kChunkBytes >> 4);
          b_lo += 2 * n;
          acc = 1;
        }
        umma_commit(&empty[rs.slot]);
      }
      __syncwarp();
      rs.next();
    }
  }
}

// ------------------------------------------------------------------------------------------------------
// positional encoding, posenc_orig (model_utils.py:234-246): [x, sin(2^k x), cos(2^k x)]_k, blocks of NC.
// sin/cos of the base angle from sincosf, higher octaves by the double-angle recurrence (fp32); the result
// is consumed as a bf16 operand, the recurrence error (<= 2^k ulp) is far below the bf16 rounding step.
// ------------------------------------------------------------------------------------------------------
template <int NC, int NF>
__device__ __forceinline__ void posenc(const float* x, float* out) {
  float s[NC], c[NC];
#pragma unroll
  for (int i = 0; i < NC; ++i) { out[i] = x[i]; sincosf(x[i], &s[i], &c[i]); }
#pragma unroll
  for (int k = 0; k < NF; ++k) {
#pragma unroll
    for (int i = 0; i < NC; ++i) {
      out[NC + 2 * NC * k + i] = s[i];
      out[NC + 2 * NC * k + NC + i] = c[i];
      float s2 = 2.f * s[i] * c[i];
      float c2 = 1.f - 2.f * s[i] * s[i];
      s[i] = s2; c[i] = c2;
    }
  }
}
// chain rule through posenc: g_x[i] = g[i] + sum_k 2^k (g_sin[k][i] cos_k - g_cos[k][i] sin_k)
template <int NC, int NF>
__device__ __forceinline__ void posenc_bwd(const float* x, const float* g, float* gx) {
  float s[NC], c[NC];
#pragma unroll
  for (int i = 0; i < NC; ++i) { gx[i] = g[i]; sincosf(x[i], &s[i], &c[i]); }
  float f = 1.f;
#pragma unroll
  for (int k = 0; k < NF; ++k) {
#pragma unroll
    for (int i = 0; i < NC; ++i) {
      gx[i] += f * (g[NC + 2 * NC * k + i] * c[i] - g[NC + 2 * NC * k + NC + i] * s[i]);
      float s2 = 2.f * s[i] * c[i];
      float c2 = 1.f - 2.f * s[i] * s[i];
      s[i] = s2; c[i] = c2;
    }
    f *= 2.f;
  }
}

// d posenc / d x[c] (the tangent of posenc along input direction c): identity column c -> 1, band k of coordinate c:
// sin column -> 2^k cos(2^k x_c), cos column -> -2^k sin(2^k x_c); every other column 0.  The sines and cosines are the
// primal's (sincosf of the base angle, double-angle recurrence), so the tangent matches the encoding it differentiates.
template <int NC, int NF>
__device__ __forceinline__ void posenc_tangent(const float* x, int c, float* out) {
#pragma unroll
  for (int i = 0; i < NC + 2 * NC * NF; ++i) out[i] = 0.f;
  float xc = 0.f;
#pragma unroll
  for (int i = 0; i < NC; ++i) if (i == c) { xc = x[i]; out[i] = 1.f; }
  float s, cs;
  sincosf(xc, &s, &cs);
  float f = 1.f;
#pragma unroll
  for (int k = 0; k < NF; ++k) {
#pragma unroll
    for (int i = 0; i < NC; ++i) {
      if (i == c) { out[NC + 2 * NC * k + i] = f * cs; out[NC + 2 * NC * k + NC + i] = -f * s; }
    }
    float s2 = 2.f * s * cs;
    float c2 = 1.f - 2.f * s * s;
    s = s2; cs = c2;
    f *= 2.f;
  }
}

// posenc_orig with a run-time frequency count nf <= NFMAX: the columns of the frequencies >= nf are zero
template <int NC, int NFMAX>
__device__ __forceinline__ void posenc_rt(const float* x, float* out, int nf) {
  float s[NC], c[NC];
#pragma unroll
  for (int i = 0; i < NC; ++i) { out[i] = x[i]; sincosf(x[i], &s[i], &c[i]); }
#pragma unroll
  for (int k = 0; k < NFMAX; ++k) {
    const bool on = k < nf;
#pragma unroll
    for (int i = 0; i < NC; ++i) {
      out[NC + 2 * NC * k + i] = on ? s[i] : 0.f;
      out[NC + 2 * NC * k + NC + i] = on ? c[i] : 0.f;
      float s2 = 2.f * s[i] * c[i];
      float c2 = 1.f - 2.f * s[i] * s[i];
      s[i] = s2; c[i] = c2;
    }
  }
}

// posenc(x, 0, NF) of SE3Field (model_utils.py:255-273): scales 2^linspace(0, NF, NF) as torch computes them in fp32 (NF = 8),
// cos as sin(x s + 0.5 * 3.1415926); per scale [sin x0..2 | "cos" x0..2], no identity columns.  Full-precision sinf: the
// arguments reach ~400 rad and the reference's shifted-sine form is only reproduced by evaluating exactly that expression.
__device__ __forceinline__ void posenc_se3(const float* x, float* out) {
  constexpr float kScale[kSe3Freqs] = {0x1.000000p+0f, 0x1.1aa59cp+1f, 0x1.381148p+2f, 0x1.588ceep+3f,
                                       0x1.7c6a1ap+4f, 0x1.a40302p+5f, 0x1.cfbb04p+6f, 0x1.000000p+8f};
#pragma unroll
  for (int k = 0; k < kSe3Freqs; ++k) {
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      const float xb = x[i] * kScale[k];
      out[6 * k + i] = sinf(xb);
      out[6 * k + 3 + i] = sinf(xb + 1.5707963f);
    }
  }
}

// se(3) exponential of the screw (w, v) applied to a point (warping.py:229-238, rigid_body.py:55-83), written with the
// un-normalised w, v so that theta -> 0 is a removable singularity:
//   y = x + v + A (w x x) + B (w x (w x x) + w x v) + C (w x (w x v)),
//   A = sin t / t, B = (1 - cos t) / t^2, C = (t - sin t) / t^3, t = |w|
// (= R x + G(t) v / t with R = I + sin t [w/t] + (1 - cos t) [w/t]^2, Modern Robotics Eq. 3.88).  Below t = 0.25 the
// coefficients and their derivative factors X'(t) / t come from their Taylor series in t^2 (next term < 1e-10).
struct Se3Coefs { float A, B, C, Ap, Bp, Cp; };
template <bool GRAD>
__device__ __forceinline__ Se3Coefs se3_coefs(float t2) {
  Se3Coefs c;
  if (t2 < 0.0625f) {
    c.A = 1.f + t2 * (-1.f / 6 + t2 * (1.f / 120 - t2 * (1.f / 5040)));
    c.B = 0.5f + t2 * (-1.f / 24 + t2 * (1.f / 720 - t2 * (1.f / 40320)));
    c.C = 1.f / 6 + t2 * (-1.f / 120 + t2 * (1.f / 5040 - t2 * (1.f / 362880)));
    if (GRAD) {
      c.Ap = -1.f / 3 + t2 * (1.f / 30 + t2 * (-1.f / 840 + t2 * (1.f / 45360)));
      c.Bp = -1.f / 12 + t2 * (1.f / 180 + t2 * (-1.f / 6720 + t2 * (1.f / 453600)));
      c.Cp = -1.f / 60 + t2 * (1.f / 1260 + t2 * (-1.f / 60480 + t2 * (1.f / 4989600)));
    }
  } else {
    const float t = sqrtf(t2), it2 = 1.f / t2;
    float sn, cs;
    sincosf(t, &sn, &cs);
    float sh, ch;
    sincosf(0.5f * t, &sh, &ch);
    c.A = sn / t;
    c.B = 2.f * sh * sh * it2;              // (1 - cos t) / t^2 without the cancellation
    c.C = (t - sn) * it2 / t;
    if (GRAD) { c.Ap = (cs - c.A) * it2; c.Bp = (c.A - 2.f * c.B) * it2; c.Cp = (c.B - 3.f * c.C) * it2; }
  }
  return c;
}
__device__ __forceinline__ void cross3(const float* a, const float* b, float* o) {
  o[0] = a[1] * b[2] - a[2] * b[1]; o[1] = a[2] * b[0] - a[0] * b[2]; o[2] = a[0] * b[1] - a[1] * b[0];
}
__device__ __forceinline__ float dot3(const float* a, const float* b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }
__device__ __forceinline__ void se3_apply(const float* x, const float* w, const float* v, float* y) {
  const Se3Coefs c = se3_coefs<false>(dot3(w, w));
  float wx[3], wwx[3], wv[3], wwv[3];
  cross3(w, x, wx); cross3(w, wx, wwx); cross3(w, v, wv); cross3(w, wv, wwv);
#pragma unroll
  for (int i = 0; i < 3; ++i) y[i] = x[i] + v[i] + c.A * wx[i] + c.B * (wwx[i] + wv[i]) + c.C * wwv[i];
}
// pull-back of g = dL/dy to the head outputs (w, v); the sample point itself takes no gradient
__device__ __forceinline__ void se3_apply_bwd(const float* x, const float* w, const float* v, const float* g, float* gw, float* gv) {
  const Se3Coefs c = se3_coefs<true>(dot3(w, w));
  float wx[3], wwx[3], wv[3], wwv[3], gxw[3], t0[3], t1[3], t2[3], t3[3], t4[3], t5[3];
  cross3(w, x, wx); cross3(w, wx, wwx); cross3(w, v, wv); cross3(w, wv, wwv);
  cross3(g, w, gxw);
  cross3(gxw, w, t0);
  cross3(x, g, t1); cross3(wx, g, t2); cross3(x, gxw, t3); cross3(v, g, t4); cross3(wv, g, t5);
  float t6[3];
  cross3(v, gxw, t6);
  float s[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) s[i] = wwx[i] + wv[i];
  const float k = c.Ap * dot3(g, wx) + c.Bp * dot3(g, s) + c.Cp * dot3(g, wwv);
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    gv[i] = g[i] + c.B * gxw[i] + c.C * t0[i];
    gw[i] = c.A * t1[i] + c.B * (t2[i] + t3[i] + t4[i]) + c.C * (t5[i] + t6[i]) + k * w[i];
  }
}

// zero padding of a K-wide input vector with IN real features; a vector that reaches INB's last chunk carries the two
// ones columns of the folded biases in its tail
template <class C, int K, int IN>
__device__ __forceinline__ void finish_features(float* f) {
#pragma unroll
  for (int i = IN; i < K; ++i) f[i] = 0.f;
  if constexpr (K / 8 == C::INB_CHUNKS) {
    static_assert(IN <= K - 2, "no room for the ones columns");
    f[K - 2] = 1.f; f[K - 1] = 1.f;
  }
}
// the ones chunk pair of INB when the vector just stored (K columns) does not reach it
template <class C, int K>
__device__ __forceinline__ void store_ones_pair(uint8_t* inb_row) {
  if constexpr (K / 8 < C::INB_CHUNKS) {
    if constexpr (K / 8 < C::INB_CHUNKS - 1) *reinterpret_cast<uint4*>(inb_row + (C::INB_CHUNKS - 2) * kChunkBytes) = make_uint4(0, 0, 0, 0);
    *reinterpret_cast<uint4*>(inb_row + (C::INB_CHUNKS - 1) * kChunkBytes) = make_uint4(0, 0, 0, 0x3F803F80u);   // bf16 1.0, 1.0
  }
}

// Stash stores are streaming (st.global.cs, evict-first): 9 GB per 1 M samples that nothing reads before the backward
// pass would otherwise push the 1.6 MB of weights every SM keeps re-reading out of L2 (measured: forward 4.99 -> 4.69 M
// cycles per CTA, the issuer's stage waits 13.8 -> 9.9 %).
__device__ __forceinline__ void stash_store(uint4* dst, const uint4& v) { __stcs(dst, v); }

// write NCOL (multiple of 8) fp32 features of one row as bf16 packets into an smem operand (and the stash)
template <int NCOL>
__device__ __forceinline__ void store_features(const float* f, uint8_t* buf_row, uint4* save_row, int save_chunk) {
#pragma unroll
  for (int q = 0; q < NCOL / 8; ++q) {
    uint4 v;
    v.x = pack_bf16(f[8 * q + 0], f[8 * q + 1]);
    v.y = pack_bf16(f[8 * q + 2], f[8 * q + 3]);
    v.z = pack_bf16(f[8 * q + 4], f[8 * q + 5]);
    v.w = pack_bf16(f[8 * q + 6], f[8 * q + 7]);
    *reinterpret_cast<uint4*>(buf_row + q * kChunkBytes) = v;
    if (save_row != nullptr) stash_store(&save_row[(save_chunk + q) * (kHalfChunkBytes / 16)], v);
  }
}

// the ones chunk pair of INB on its own (trunk-only rows of a model whose trunk input lives in ACT)
template <class C>
__device__ __forceinline__ void store_ones_only(uint8_t* inb_row) {
  *reinterpret_cast<uint4*>(inb_row + (C::INB_CHUNKS - 2) * kChunkBytes) = make_uint4(0, 0, 0, 0);
  *reinterpret_cast<uint4*>(inb_row + (C::INB_CHUNKS - 1) * kChunkBytes) = make_uint4(0, 0, 0, 0x3F803F80u);   // bf16 1.0, 1.0
}

// Trunk input vector of the template (models.py:458-478): [posenc_orig(xyz, XF) | posenc_orig(hyper, HF) | 0], written as
// bf16 into INB, or into ACT[0, KT) for the wide vectors (hn_mlp_program.h: kMaxTrunkInInb), and into the stash.
template <class C>
__device__ __forceinline__ void store_trunk_input(const float* wp, uint8_t* act_row, uint8_t* inb_row, uint4* save_row, int save_chunk) {
  float f[C::KT];
  posenc<3, C::XF>(wp, f);
  if constexpr (C::H > 0) posenc<C::H, C::HF>(wp + 3, f + C::PE_X);
  if constexpr (C::TIN_ACT) {
#pragma unroll
    for (int i = C::IN_T; i < C::KT; ++i) f[i] = 0.f;
    store_features<C::KT>(f, act_row, save_row, save_chunk);
  } else {
    finish_features<C, C::KT, C::IN_T>(f);
    store_features<C::KT>(f, inb_row, save_row, save_chunk);
  }
}

// Warp-stage input vector of SE3 + sheet (Shape::WS_ACT): [posenc(points, 0, WF) | posenc_orig(points, SF) | GLO | 0],
// written as bf16 into ACT[0, KW) (and the stash) by the prologue, and again by the FE_SKIPFEED epilogue
template <class C>
__device__ __forceinline__ void store_ws_input(const FwdParams& p, int64_t gq, int64_t ray, uint8_t* act_row, uint4* save_row,
                                               int save_chunk) {
  float f[C::KW], pt[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) pt[i] = __ldg(p.points + gq * 3 + i);
  posenc_se3(pt, f);
  posenc<3, C::SF>(pt, f + C::PE_W);
  const int64_t id = __ldg(p.ids + ray);
  HN_CHECK_ID(id, p.n_embed);
  const float* e = p.glo + id * C::G;
#pragma unroll
  for (int i = 0; i < C::G; ++i) f[C::PE_W + C::PE_S + i] = __ldg(e + i);
#pragma unroll
  for (int i = C::IN_W; i < C::KW; ++i) f[i] = 0.f;
  store_features<C::KW>(f, act_row, save_row, save_chunk);
}

// d(GLO embedding) of one sample (G values in r[0..G)) -> per-ray reduction -> atomics on the table gradient
template <int G>
__device__ __forceinline__ void glo_grad_add(const float* v_in, bool valid, int64_t id, float* __restrict__ glo_grad, int lane) {
  const bool uniform = __all_sync(0xffffffffu, id == __shfl_sync(0xffffffffu, id, 0));
#pragma unroll
  for (int i = 0; i < G; ++i) {
    float v = valid ? v_in[i] : 0.f;
    if (uniform) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) atomicAdd(glo_grad + id * G + i, v);
    } else {
      atomicAdd(glo_grad + id * G + i, v);
    }
  }
}

// ------------------------------------------------------------------------------------------------------
// generic epilogue column loops: this thread's row of the accumulator, 32 columns at a time, TMEM loads
// double-buffered (the load of block b+1 is in flight while block b is converted and stored).
// ------------------------------------------------------------------------------------------------------
// One mbarrier arrival per warp instead of 32: every lane has fenced its own writes, __syncwarp orders them before
// lane 0's (release) arrive.  256 individual arrivals on one shared-memory word serialise for several hundred cycles on
// the critical path between a layer's epilogue and the next layer's first UMMA.
__device__ __forceinline__ void warp_arrive(uint64_t* bar) {
  __syncwarp();
  if ((threadIdx.x & 31) == 0) mbar_arrive(bar);
}
// named barrier of one chain's epilogue threads (ids 1, 2; barrier 0 is __syncthreads)
template <bool PP>
__device__ __forceinline__ void epi_named_barrier(int chain) {
  asm volatile("bar.sync %0, %1;" ::"r"(1 + chain), "n"(128 * Sched<PP>::SUBS * kEpiSplit) : "memory");
}

// bias of a head column: FOLD = already inside the accumulator (bias K steps), else from the shared-memory staging buffer
template <bool FOLD>
__device__ __forceinline__ float head_bias(const float* bias_s, int i) {
  return FOLD ? 0.f : bias_s[i];
}

// one 32-column block (4 chunks of 8 columns): bias, ReLU, bf16 pack, st.shared (+ stash store and gate word: the sign
// bits of the even / odd columns, hn_ptx.cuh: gate_push)
template <bool RELU, bool STASH, bool FOLD>
__device__ __forceinline__ void fwd_store32(const uint32_t* r, const float* bias_s, uint8_t* act_row, uint4* save_row,
                                            int chunk0, int save_chunk, uint32_t* gate_dst) {
  uint32_t ge = 0, go = 0;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    float v[8];
    if constexpr (FOLD) {   // the accumulator already holds W x + b
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = __uint_as_float(r[8 * q + j]);
    } else {                // smem broadcast
    const float4 b0 = *reinterpret_cast<const float4*>(bias_s + 8 * q);
    const float4 b1 = *reinterpret_cast<const float4*>(bias_s + 8 * q + 4);
    v[0] = __uint_as_float(r[8 * q + 0]) + b0.x; v[1] = __uint_as_float(r[8 * q + 1]) + b0.y;
    v[2] = __uint_as_float(r[8 * q + 2]) + b0.z; v[3] = __uint_as_float(r[8 * q + 3]) + b0.w;
    v[4] = __uint_as_float(r[8 * q + 4]) + b1.x; v[5] = __uint_as_float(r[8 * q + 5]) + b1.y;
    v[6] = __uint_as_float(r[8 * q + 6]) + b1.z; v[7] = __uint_as_float(r[8 * q + 7]) + b1.w;
    }
    uint4 o;
    if (RELU) {
      o.x = pack_bf16_relu(v[0], v[1]); o.y = pack_bf16_relu(v[2], v[3]);
      o.z = pack_bf16_relu(v[4], v[5]); o.w = pack_bf16_relu(v[6], v[7]);
      if (STASH) {
#pragma unroll
        for (int j = 0; j < 4; ++j) { ge = gate_push(ge, v[2 * j]); go = gate_push(go, v[2 * j + 1]); }
      }
    } else {
      o.x = pack_bf16(v[0], v[1]); o.y = pack_bf16(v[2], v[3]);
      o.z = pack_bf16(v[4], v[5]); o.w = pack_bf16(v[6], v[7]);
    }
    *reinterpret_cast<uint4*>(act_row + (chunk0 + q) * kChunkBytes) = o;
    if (STASH) stash_store(&save_row[(save_chunk + chunk0 + q) * (kHalfChunkBytes / 16)], o);
  }
  if (RELU && STASH) __stcs(&gate_dst[(chunk0 >> 2) * kHalfRows], gate_word_of(ge, go));
}

// ncols: multiple of 32
template <bool RELU, bool STASH, bool FOLD>
__device__ __forceinline__ void fwd_cols(uint32_t taddr, const float* bias_s, uint8_t* act_row, uint4* save_row,
                                         int save_chunk, int ncols, uint32_t* gate_dst) {
  if constexpr (kEpiSplit == 2) {
    // two warpgroups per sub-tile overlap each other's TMEM latency: one buffer keeps the secondary warpgroup at 64 registers
    uint32_t r[32];
    for (int c0 = 0; c0 < ncols; c0 += 32) {
      tmem_ld32(taddr + c0, r);
      tmem_ld_wait();
      fwd_store32<RELU, STASH, FOLD>(r, bias_s + c0, act_row, save_row, c0 >> 3, save_chunk, gate_dst);
    }
    return;
  }
  uint32_t ra[32], rb[32];
  tmem_ld32(taddr, ra);
  for (int c0 = 0; c0 < ncols; c0 += 64) {
    tmem_ld_wait();
    const bool more = c0 + 32 < ncols;
    if (more) tmem_ld32(taddr + c0 + 32, rb);
    fwd_store32<RELU, STASH, FOLD>(ra, bias_s + c0, act_row, save_row, c0 >> 3, save_chunk, gate_dst);
    if (more) {
      tmem_ld_wait();
      if (c0 + 64 < ncols) tmem_ld32(taddr + c0 + 64, ra);
      fwd_store32<RELU, STASH, FOLD>(rb, bias_s + c0 + 32, act_row, save_row, (c0 + 32) >> 3, save_chunk, gate_dst);
    }
  }
}

// the column share of one of the kEpiSplit warpgroups that drain a sub-tile (hn_mlp_program.h: kEpiSplit)
template <bool RELU, bool STASH, bool FOLD>
__device__ __forceinline__ void fwd_cols_share(int share, uint32_t taddr, const float* bias_s, uint8_t* act_row,
                                               uint4* save_row, int save_chunk, int ncols, uint32_t* gate_dst) {
  const int n = ncols / kEpiSplit, c0 = share * n;
  fwd_cols<RELU, STASH, FOLD>(taddr + c0, bias_s + c0, act_row + (c0 >> 3) * kChunkBytes, save_row,
                              save_chunk + (c0 >> 3), n, gate_dst != nullptr ? gate_dst + (c0 >> 5) * kHalfRows : nullptr);
}

// backward: ReLU gates from the gate words the forward wrote (one uint32 per row per 32 columns, hn_ptx.cuh), so the
// data gradient never re-reads the 8.6 KB/sample activation stash.  The words of a layer (<= 8 per row) are requested
// before the epilogue waits for the accumulator; the packed gradient pair j of a block is masked with 3 integer ops.
template <int NCOLS>
__device__ __forceinline__ void load_gates(const uint32_t* __restrict__ gate_row, int gate_word, uint32_t* gw) {
#pragma unroll
  for (int b = 0; b < NCOLS / 32; ++b) gw[b] = __ldg(gate_row + (size_t)(gate_word + b) * kHalfRows);
}

// one 32-column block: r = accumulator row slice, w = the block's gate word
template <bool MASK>
__device__ __forceinline__ void bwd_store32(const uint32_t* r, uint32_t w, uint8_t* dst_row, uint4* save_row, int chunk0,
                                            int save_chunk) {
  uint32_t o[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) o[j] = pack_bf16(__uint_as_float(r[2 * j]), __uint_as_float(r[2 * j + 1]));
  if (MASK) {
    o[0] &= ~gate_pair_closed<0>(w); o[1] &= ~gate_pair_closed<1>(w); o[2] &= ~gate_pair_closed<2>(w); o[3] &= ~gate_pair_closed<3>(w);
    o[4] &= ~gate_pair_closed<4>(w); o[5] &= ~gate_pair_closed<5>(w); o[6] &= ~gate_pair_closed<6>(w); o[7] &= ~gate_pair_closed<7>(w);
    o[8] &= ~gate_pair_closed<8>(w); o[9] &= ~gate_pair_closed<9>(w); o[10] &= ~gate_pair_closed<10>(w); o[11] &= ~gate_pair_closed<11>(w);
    o[12] &= ~gate_pair_closed<12>(w); o[13] &= ~gate_pair_closed<13>(w); o[14] &= ~gate_pair_closed<14>(w); o[15] &= ~gate_pair_closed<15>(w);
  }
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const uint4 v = make_uint4(o[4 * q], o[4 * q + 1], o[4 * q + 2], o[4 * q + 3]);
    *reinterpret_cast<uint4*>(dst_row + (chunk0 + q) * kChunkBytes) = v;
    if (save_row != nullptr) stash_store(&save_row[(save_chunk + chunk0 + q) * (kHalfChunkBytes / 16)], v);
  }
}
// NCOLS: multiple of 32 (<= 256), compile time so that gw[] and both row buffers stay in registers
template <bool MASK, int NCOLS>
__device__ __forceinline__ void bwd_cols(uint32_t taddr, const uint32_t* gw, uint8_t* dst_row, uint4* save_row, int save_chunk) {
  if constexpr (kEpiSplit == 2) {
    uint32_t r[32];
#pragma unroll
    for (int b = 0; b < NCOLS / 32; ++b) {
      tmem_ld32(taddr + b * 32, r);
      tmem_ld_wait();
      bwd_store32<MASK>(r, MASK ? gw[b] : 0u, dst_row, save_row, b * 4, save_chunk);
    }
    return;
  }
  uint32_t r[2][32];
  tmem_ld32(taddr, r[0]);
#pragma unroll
  for (int b = 0; b < NCOLS / 32; ++b) {
    tmem_ld_wait();
    if (b + 1 < NCOLS / 32) tmem_ld32(taddr + (b + 1) * 32, r[(b + 1) & 1]);
    bwd_store32<MASK>(r[b & 1], MASK ? gw[b] : 0u, dst_row, save_row, b * 4, save_chunk);
  }
}
// masked layer of width NCOLS: gate fetch, accumulator wait, masked store
template <int NCOLS>
__device__ __forceinline__ void bwd_masked_layer(uint32_t tlane, const uint32_t* __restrict__ gate_row, int gate_word, uint8_t* dst_row,
                                                 uint4* save_row, int save_chunk, uint64_t* acc_full, uint32_t& ph_acc, long long& t_acc) {
  uint32_t gw[NCOLS / 32];
  load_gates<NCOLS>(gate_row, gate_word, gw);
  { long long t0 = HN_T0(); mbar_wait(acc_full, ph_acc); ph_acc ^= 1; t_acc += HN_T0() - t0; }
  tc_fence_after();
  bwd_cols<true, NCOLS>(tlane, gw, dst_row, save_row, save_chunk);
}

// the column share of one of the kEpiSplit warpgroups of a sub-tile (hn_mlp_program.h: kEpiSplit)
template <int NCOLS>
__device__ __forceinline__ void bwd_masked_share(int share, uint32_t tlane, const uint32_t* __restrict__ gate_row, int gate_word,
                                                 uint8_t* dst_row, uint4* save_row, int save_chunk, uint64_t* acc_full,
                                                 uint32_t& ph_acc, long long& t_acc) {
  constexpr int N = NCOLS / kEpiSplit;
  const int c0 = share * N;
  bwd_masked_layer<N>(tlane + c0, gate_row, gate_word + (c0 >> 5), dst_row + (c0 >> 3) * kChunkBytes, save_row,
                      save_chunk + (c0 >> 3), acc_full, ph_acc, t_acc);
}
template <int NCOLS>
__device__ __forceinline__ void bwd_linear_share(int share, uint32_t tlane, uint8_t* dst_row, uint4* save_row, int save_chunk) {
  constexpr int N = NCOLS / kEpiSplit;
  const int c0 = share * N;
  bwd_cols<false, N>(tlane + c0, nullptr, dst_row + (c0 >> 3) * kChunkBytes, save_row, save_chunk + (c0 >> 3));
}

__device__ __forceinline__ float softplus_f(float x) { return x > 20.f ? x : log1pf(expf(x)); }
__device__ __forceinline__ float sigmoid_f(float x) { return 1.f / (1.f + expf(-x)); }

// ======================================================================================================
// forward
// ======================================================================================================
// tangent launch (FwdParams::jac): tile -> (input direction, primal tile) over 3 x the primal's tiles; every direction
// reads the primal tile's gate words
__device__ __forceinline__ int tangent_plane(int tile, int n_tiles) { return tile / (n_tiles / 3); }

// STASH = false (inference, hn_mlp_fwd with saved == NULL) compiles every stash store out: even predicated-off
// st.global instructions in the drain loop cost 23 % of the kernel (2.67 -> 2.06 ms per 1 M samples, measured).
// TANGENT (with STASH, translation warp only): the program is ModelPlan::fwd_warp_tangent, one launch for the three input
// directions (FwdParams::jac); its stash stores are skipped at run time when FwdParams::saved is NULL.
template <class C, bool STASH, bool TANGENT = false>
__global__ void __launch_bounds__(kMlpThreads, 1) mlp_fwd_kernel(const __grid_constant__ FwdParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  using SM = Smem<C>;
  // biases inside the UMMAs in inference (hn_mlp_program.h: bias folding), staged in smem by the stash-writing forward
  constexpr bool FOLD = !STASH;
  constexpr bool PP = STASH;   // out of phase in training, lock step in inference (see Sched)
  uint8_t* act = smem + SM::ACT;
  uint8_t* inb = smem + SM::INB;
  uint8_t* ring = smem + SM::RING;
  float* sbias = reinterpret_cast<float*>(smem + SM::BIAS);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + SM::BARS);
  uint64_t* empty = full + kRingStages;
  uint64_t* acc_full = empty + kRingStages;   // [2]: one per chain
  uint64_t* act_ready = acc_full + 2;         // [2]
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(smem + SM::TMEMP);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int i = 0; i < kRingStages; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    // one arrival per epilogue warp of the chain
    for (int i = 0; i < 2; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&act_ready[i], 4 * Sched<PP>::SUBS * kEpiSplit); }
    fence_barrier_init();
  }
  if (warp == kIssuerWarp) { tmem_alloc(tmem_ptr, 256 * kSubTiles); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  const Program& prog = p.prog;

  if (warp >= kEpiWarps) {
    setmaxnreg_dec<kRegsFeeder>();
    if (warp == kProducerWarp && lane == 0) {
      RingState rs;
      long long tw = 0;
      for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) produce_tile<PP>(prog, p.weights, ring, full, empty, rs, tw);
      if (p.dbg) p.dbg[blockIdx.x * 8 + 0] = tw;
    } else if (warp == kIssuerWarp) {  // whole warp, converged: see elect_one_sync()
      RingState rs;
      uint32_t ph_ready = 0;
      long long t_ready = 0, t_full = 0;
      const long long t_begin = HN_T0();
      const uint32_t act_s = smem_u32(act), inb_s = smem_u32(inb), ring_s = smem_u32(ring);
      for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
        for (int li = 0; li < prog.nlayers; ++li) {
          for (int chain = 0; chain < Sched<PP>::CHAINS; ++chain) {
            long long t0 = HN_T0();
            mbar_wait(&act_ready[chain], ph_ready);
            t_ready += HN_T0() - t0;
            tc_fence_after();
            issue_layer<PP>(prog, prog.layers[li], chain * Sched<PP>::SUBS, act_s, inb_s, SM::ACT_BYTES, SM::INB_BYTES, ring_s, tmem_base,
                        full, empty, rs, t_full);
            if (elect_one_sync()) umma_commit(&acc_full[chain]);
            __syncwarp();
          }
          ph_ready ^= 1;
        }
      }
      if (p.dbg && lane == 0) {
        p.dbg[blockIdx.x * 8 + 1] = t_ready; p.dbg[blockIdx.x * 8 + 2] = t_full; p.dbg[blockIdx.x * 8 + 3] = HN_T0() - t_begin;
      }
    }
  } else {
    // ---------------- epilogue warps: thread <-> sample row; kEpiSplit warpgroups per sub-tile ----------------
    const int et = threadIdx.x % (128 * Sched<PP>::SUBS * kEpiSplit);  // index inside this chain's epilogue threads
    const int sub = warp / (4 * kEpiSplit);
    const int share = (warp >> 2) % kEpiSplit;   // which column share of the wide drains; share 0 = the primary warpgroup
    const int quarter = warp & 3;            // TMEM lane quarter this warp may access
    auto epilogue = [&](auto primary_tag) {
    constexpr bool PRIMARY = decltype(primary_tag)::value;   // primary: per-row work (encodings, heads) + its column share
    const int row = quarter * 32 + lane;     // row inside the sub-tile
    const uint32_t tlane = tmem_base + ((uint32_t)(quarter * 32) << 16) + sub * 256;
    uint8_t* act_row = act + sub * SM::ACT_BYTES + row * 16;
    uint8_t* inb_row = inb + sub * SM::INB_BYTES + row * 16;
    const int chain = PP ? sub : 0;
    uint64_t* my_acc = &acc_full[chain];
    uint64_t* my_ready = &act_ready[chain];
    uint32_t ph_acc = 0;
    long long t_acc = 0, t_pro = 0;
    const long long t_begin = HN_T0();
    for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
      const long long t_tile = HN_T0();
      const int64_t g = (int64_t)(TANGENT ? tile % (p.n_tiles / 3) : tile) * kCtaRows + sub * kTileRows + row;
      const bool valid = g < p.n;
      const int64_t gc = valid ? g : p.n - 1;
      const int64_t ray = gc / p.S;
      // where this row lives in the caller's (B, S_full) tensors (points, noise, sigma, rgb, warped)
      const int64_t gq = p.pos != nullptr ? ray * p.S_full + __ldg(p.pos + gc) : gc;
      uint4* save_row = nullptr;
      uint32_t* gate_row = nullptr;   // this row's column of the half tile's gate words
      if constexpr (TANGENT) {
        const size_t half = (size_t)(tile % (p.n_tiles / 3)) * (2 * kSubTiles) + sub * 2 + (row >> 6);
        gate_row = p.gates + half * (size_t)p.g_total * kHalfRows + (row & 63);
        if (p.saved != nullptr) {   // plane c of the tangent stash: the warp-only stash layout of the primal's tiles
          const size_t plane_bytes = (size_t)(p.n_tiles / 3) * (2 * kSubTiles) * ((size_t)p.x_total * kHalfChunkBytes + (size_t)p.g_total * kHalfRows * 4);
          save_row = reinterpret_cast<uint4*>(p.saved + tangent_plane(tile, p.n_tiles) * plane_bytes +
                                              half * (size_t)p.x_total * kHalfChunkBytes) + (row & 63);
        }
      } else if (p.saved != nullptr) {
        const size_t half = (size_t)tile * (2 * kSubTiles) + sub * 2 + (row >> 6);
        save_row = reinterpret_cast<uint4*>(p.saved + half * (size_t)p.x_total * kHalfChunkBytes) + (row & 63);
        gate_row = p.gates + half * (size_t)p.g_total * kHalfRows + (row & 63);
      }
      // (the sample point and view direction are re-loaded where they are needed — FE_WSHEAD, FE_BOTT — instead of being
      // kept in registers across the drain loops; only the wide trunk inputs keep the warped point for FE_SKIPFEED)
      float wp_keep[C::TIN_ACT ? C::NWARPED : 1];
      float hy_keep[C::WS_ACT ? C::H : 1];   // SE3 + sheet: the sheet's hyper coordinates, from FE_LINSHEET to FE_WSHEAD
      const bool trunk_only = !C::STATIC && p.warped_in != nullptr;
      if constexpr (PRIMARY && TANGENT) {
        // prologue: d posenc(points, WF) / d x[plane] | 0 (GLO columns and padding) -> INB and the tangent stash
        float f[C::KW], pt[3];
#pragma unroll
        for (int i = 0; i < 3; ++i) pt[i] = __ldg(p.points + gq * 3 + i);
        posenc_tangent<3, C::WF>(pt, tangent_plane(tile, p.n_tiles), f);
#pragma unroll
        for (int i = C::PE_W; i < C::KW; ++i) f[i] = 0.f;
        store_features<C::KW>(f, inb_row, save_row, p.x_in_ws);
      } else if constexpr (PRIMARY) {
      if (trunk_only) {
        // trunk-only program: the warped point / hyper coordinates of this row were computed by another launch (the
        // coarse level's, for the depths the fine level inherits) or are the raw sample point (model without warp); the
        // prologue does what FE_WSHEAD's epilogue does
        if constexpr (!C::STATIC) {
          float wp[C::NWARPED];
#pragma unroll
          for (int i = 0; i < C::NWARPED; ++i) wp[i] = __ldg(p.warped_in + gc * C::NWARPED + i);
          if (valid && p.warped != nullptr) {   // the given point is also this row's entry of the level's warped_points
#pragma unroll
            for (int i = 0; i < C::NWARPED; ++i) p.warped[gq * C::NWARPED + i] = wp[i];
          }
          store_trunk_input<C>(wp, act_row, inb_row, save_row, p.x_in_t);
          if constexpr (C::TIN_ACT) {
            store_ones_only<C>(inb_row);
#pragma unroll
            for (int i = 0; i < C::NWARPED; ++i) wp_keep[i] = wp[i];
          } else {
            store_ones_pair<C, C::KT>(inb_row);
          }
        }
      } else if constexpr (C::WS_ACT) {
        // prologue: the warp-stage vector -> ACT; INB only gets the ones pair of the folded biases (the trunk input follows
        // from FE_WSHEAD)
        store_ws_input<C>(p, gq, ray, act_row, save_row, p.x_in_ws);
        store_ones_only<C>(inb_row);
      } else if constexpr (!C::NOWARP) {
      // prologue: [posenc(points, WF) | GLO | 0] -> INB   (static baseline: [Embedding(xyz) | 0], nerf.py:21-38)
        float f[C::KW];
        {
          float pt[3];
#pragma unroll
          for (int i = 0; i < 3; ++i) pt[i] = __ldg(p.points + gq * 3 + i);
          if constexpr (C::SE3) posenc_se3(pt, f); else posenc<3, C::WF>(pt, f);
        }
        if constexpr (!C::STATIC && !C::SE3) {
          const int64_t id = __ldg(p.ids + ray);
          HN_CHECK_ID(id, p.n_embed);   // out-of-range metadata id
          const float* e = p.glo + id * C::G;
#pragma unroll
          for (int i = 0; i < C::G; ++i) f[C::PE_W + i] = __ldg(e + i);
        }
        finish_features<C, C::KW, C::IN_W>(f);
        store_features<C::KW>(f, inb_row, save_row, p.x_in_ws);
        store_ones_pair<C, C::KW>(inb_row);
      }
      }   // PRIMARY
      fence_proxy_async_smem();
      tc_fence_before();
      warp_arrive(my_ready);
      t_pro += HN_T0() - t_tile;

      for (int li = 0; li < prog.nlayers; ++li) {
        const Layer& L = prog.layers[li];
        // stage this layer's bias in shared memory while the MMAs run (L1 is ~0 KB at this smem carve-out,
        // a per-block __ldg would go to L2 every time); double-buffered by layer parity
        float* bias = PP ? sbias + chain * 256 : sbias + (li & 1) * 256;
        const long long t_layer = HN_T0();
        if constexpr (!FOLD && !TANGENT) {
          if (PP) epi_named_barrier<PP>(chain);   // single buffer per chain: everyone is done with the previous layer's bias
          for (int i = et; i < L.n_out; i += 128 * Sched<PP>::SUBS * kEpiSplit) bias[i] = __ldg(p.bias + L.bias_off + i);
          epi_named_barrier<PP>(chain);
        }
        { long long t0 = HN_T0(); mbar_wait(my_acc, ph_acc); ph_acc ^= 1; t_acc += HN_T0() - t0; }
        tc_fence_after();
        const long long t_drain = HN_T0();
        if constexpr (TANGENT) {
          if (L.epi == FE_TANGENT) {
            // D_l W_l t_{l-1}: the bf16 tangent masked by the primal's ReLU gates, into ACT and the tangent stash
            uint32_t gw[kWsW / 32];
            load_gates<kWsW>(gate_row, L.gate_word, gw);
            bwd_cols<true, kWsW>(tlane, gw, act_row, save_row, L.save_chunk);
          } else if constexpr (PRIMARY) {   // FE_JACHEAD
            uint32_t r[16];
            tmem_ld16(tlane, r);
            tmem_ld_wait();
            const int plane = tangent_plane(tile, p.n_tiles);
            if (valid) {
#pragma unroll
              for (int i = 0; i < 3; ++i) p.jac[gq * 9 + i * 3 + plane] = __uint_as_float(r[i]) + (i == plane ? 1.f : 0.f);
            }
          }
        } else if (L.epi == FE_RELU) {
          fwd_cols_share<true, STASH, FOLD>(share, tlane, bias, act_row, save_row, L.save_chunk, L.n_out,
                                      STASH ? gate_row + (size_t)L.gate_word * kHalfRows : nullptr);
        } else if (L.epi == FE_WSHEAD) {
          if constexpr (PRIMARY && !C::STATIC && !C::NOWARP) {
          uint32_t r[16];
          tmem_ld16(tlane, r);
          float wp[C::NWARPED];
#pragma unroll
          for (int i = 0; i < 3; ++i) wp[i] = __ldg(p.points + gq * 3 + i);
          tmem_ld_wait();
          if constexpr (C::SE3) {
            // head columns 0..2 = w, 3..5 = v: rigid transform of the sample point by exp of the screw (warping.py:229-238)
            float wv[6], x[3];
#pragma unroll
            for (int i = 0; i < 6; ++i) wv[i] = __uint_as_float(r[i]) + head_bias<FOLD>(bias, i);
#pragma unroll
            for (int i = 0; i < 3; ++i) x[i] = wp[i];
            se3_apply(x, wv, wv + 3, wp);
            if constexpr (C::WS_ACT) {
#pragma unroll
              for (int i = 0; i < C::H; ++i) wp[3 + i] = hy_keep[i];
            }
            if (valid && p.aux != nullptr) {
#pragma unroll
              for (int i = 0; i < 6; ++i) p.aux[g * 6 + i] = wv[i];
            }
          } else {
#pragma unroll
          for (int i = 0; i < 3; ++i) wp[i] += __uint_as_float(r[i]) + head_bias<FOLD>(bias, i);
#pragma unroll
          for (int i = 0; i < C::H; ++i) wp[3 + i] = __uint_as_float(r[3 + i]) + head_bias<FOLD>(bias, 3 + i);
          }
          if constexpr (C::H == C::G) {
            if (p.mflags & MF_AXIS) {   // axis-aligned slicing: the hyper point is the GLO vector (models.py:533-534)
              const int64_t id = __ldg(p.ids + ray);
              HN_CHECK_ID(id, p.n_embed);
              const float* e = p.glo + id * C::G;
#pragma unroll
              for (int i = 0; i < C::G; ++i) wp[3 + i] = __ldg(e + i);
            }
          }
          if (valid && p.warped != nullptr) {
#pragma unroll
            for (int i = 0; i < C::NWARPED; ++i) p.warped[gq * C::NWARPED + i] = wp[i];
          }
          // a warp-stage-only program ends here: no trunk input (its stash has no slab for it)
          if (!(prog.flags & PF_WARP_ONLY)) {
            store_trunk_input<C>(wp, act_row, inb_row, save_row, L.save_chunk);
            if constexpr (C::TIN_ACT) {
#pragma unroll
              for (int i = 0; i < C::NWARPED; ++i) wp_keep[i] = wp[i];
            }
          }
          }
        } else if (L.epi == FE_SKIPFEED) {
          // hidden part of the skip layer is in the accumulator and stays there; ACT[0, KT) <- the trunk input vector,
          // recomputed from the warped point this thread still holds, for the input part that accumulates on top
          // (SE3 + sheet: the warp stage's skip layer, ACT[0, KW) <- the warp-stage vector)
          if constexpr (PRIMARY && C::TIN_ACT) store_trunk_input<C>(wp_keep, act_row, inb_row, nullptr, 0);
          if constexpr (PRIMARY && C::WS_ACT) store_ws_input<C>(p, gq, ray, act_row, nullptr, 0);
        } else if (L.epi == FE_LINEAR) {
          fwd_cols_share<false, STASH, FOLD>(share, tlane, bias, act_row, save_row, L.save_chunk, L.n_out, nullptr);
        } else if (C::WS_ACT && L.epi == FE_LINSHEET) {
          // SE3 logit columns [0, 128) as FE_LINEAR; the sheet's H outputs in [128, 144) are kept for FE_WSHEAD
          fwd_cols_share<false, STASH, FOLD>(share, tlane, bias, act_row, save_row, L.save_chunk, kSe3W, nullptr);
          if constexpr (PRIMARY && C::WS_ACT) {
            uint32_t r[16];
            tmem_ld16(tlane + kSe3W, r);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < C::H; ++i) hy_keep[i] = __uint_as_float(r[i]) + head_bias<FOLD>(bias, kSe3W + i);
          }
        } else if (L.epi == FE_SIGMA) {
          // static baseline: raw sigma = Linear(W, 1)(h8) (nerf.py:109); rendering.py:150 uses relu(sigma + noise)
          if constexpr (PRIMARY) {
          uint32_t r[16];
          tmem_ld16(tlane, r);
          tmem_ld_wait();
          float a = __uint_as_float(r[0]) + head_bias<FOLD>(bias, 0);
          if (p.noise != nullptr) a += __ldg(p.noise + gq) * p.noise_std;
          if (valid) p.sigma[gq] = fmaxf(a, 0.f);
          }
        } else if (L.epi == FE_BOTT) {
          fwd_cols_share<false, STASH, FOLD>(share, tlane, bias, act_row, save_row, L.save_chunk, L.n_out, nullptr);
          // view-direction condition (models.py:410-419; viewdirs = raw directions, models.py:717-720)
          if constexpr (PRIMARY) {
          float f[C::KV], dir[3];
#pragma unroll
          for (int i = 0; i < 3; ++i) dir[i] = __ldg(p.viewdirs + ray * 3 + i);
          if constexpr (C::STATIC) {
            posenc<3, C::VF>(dir, f);
            finish_features<C, C::KV, C::PE_V>(f);
          } else {
            // [posenc_orig(viewdirs, view_freqs) | 0 .. | GLO condition] (hn_mlp_program.h: kViewCondCol)
            posenc_rt<3, kMaxViewFreqs>(dir, f, p.view_freqs);
#pragma unroll
            for (int i = 3 + 6 * kMaxViewFreqs; i < C::KV; ++i) f[i] = 0.f;
            if (p.mflags & MF_COND) {   // get_condition_inputs, models.py:421-434
              const int64_t id = __ldg(p.ids + ray);
              HN_CHECK_ID(id, p.n_embed);
              const float* e = p.glo + id * C::G;
#pragma unroll
              for (int i = 0; i < C::G; ++i) f[kViewCondCol + i] = __ldg(e + i);
            }
          }
          store_features<C::KV>(f, inb_row, save_row, p.x_in_v);
          }
        } else if (L.epi == FE_RGB0A) {
          if constexpr (!C::STATIC) {
          fwd_cols_share<true, STASH, FOLD>(share, tlane, bias, act_row, save_row, L.save_chunk, kRgbW,
                                      STASH ? gate_row + (size_t)L.gate_word * kHalfRows : nullptr);
          if constexpr (PRIMARY) {
          uint32_t r[16];
          tmem_ld16(tlane + kRgbW, r);
          tmem_ld_wait();
          float a = __uint_as_float(r[0]) + head_bias<FOLD>(bias, kRgbW);
          if (p.noise != nullptr) a += __ldg(p.noise + gq) * p.noise_std;  // noise_regularize, model_utils.py:312-316
          if (valid) p.sigma[gq] = softplus_f(a);                         // models.py:491
          }
          }
        } else if constexpr (PRIMARY) {  // FE_RGBHEAD
          uint32_t r[16];
          tmem_ld16(tlane, r);
          tmem_ld_wait();
          if (valid) {
#pragma unroll
            for (int i = 0; i < 3; ++i) p.rgb[gq * 3 + i] = sigmoid_f(__uint_as_float(r[i]) + head_bias<FOLD>(bias, i));
          }
        }
        if (li + 1 < prog.nlayers) {
          fence_proxy_async_smem();
          tc_fence_before();
          warp_arrive(my_ready);
        }
#if HN_ROLE_TIMING
        // per-layer profile of CTA 0 (profiles/role_timing.py): [wait for the accumulator, drain] after the 8 role counters
        if (p.dbg && blockIdx.x == 0 && threadIdx.x == 0) {
          p.dbg[gridDim.x * 8 + li * 2] += t_drain - t_layer;
          p.dbg[gridDim.x * 8 + li * 2 + 1] += HN_T0() - t_drain;
        }
#endif
        (void)t_layer; (void)t_drain;
      }
    }
    if (p.dbg && threadIdx.x == 0) {
      const long long tt = HN_T0() - t_begin;
      p.dbg[blockIdx.x * 8 + 4] = t_acc; p.dbg[blockIdx.x * 8 + 5] = tt - t_acc - t_pro;
      p.dbg[blockIdx.x * 8 + 6] = t_pro; p.dbg[blockIdx.x * 8 + 7] = tt;
    }
    };   // epilogue
    // the two kinds of epilogue warpgroups get their own register budgets (setmaxnreg is per warpgroup)
    if (kEpiSplit == 1 || share == 0) { setmaxnreg_inc<kRegsPrimary>(); epilogue(std::true_type{}); }
    else { setmaxnreg_dec<kRegsSecondary>(); epilogue(std::false_type{}); }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kIssuerWarp) tmem_dealloc(tmem_base, 256 * kSubTiles);
}

// d(trunk input features) in this row's accumulator columns [0, KT) -> d(warped point, hyper coordinates) through the
// chain rule of posenc_orig.  The wide vectors (hyper_dim 4 / 8) are consumed in two phases so that no more than ~120
// accumulator values are live at a time: columns [0, 64) = the xyz block and the first hyper column, then the rest.
template <class C>
__device__ __forceinline__ void trunk_in_bwd(uint32_t tlane, const float* wp, float* gx) {
  if constexpr (C::KT <= 96) {
    float gf[C::KT];
#pragma unroll
    for (int c0 = 0; c0 < C::KT; c0 += 32) {
      uint32_t r[32];
      tmem_ld32(tlane + c0, r);
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 32; ++j) gf[c0 + j] = __uint_as_float(r[j]);
    }
    posenc_bwd<3, C::XF>(wp, gf, gx);
    if constexpr (C::H > 0) posenc_bwd<C::H, C::HF>(wp + 3, gf + C::PE_X, gx + 3);
  } else {
    static_assert(C::PE_X == 63, "the two-phase pull-back assumes the hyper block starts at column 63");
    float gh[C::PE_H + 8];
    {
      float ga[64];
#pragma unroll
      for (int c0 = 0; c0 < 64; c0 += 32) {
        uint32_t r[32];
        tmem_ld32(tlane + c0, r);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) ga[c0 + j] = __uint_as_float(r[j]);
      }
      posenc_bwd<3, C::XF>(wp, ga, gx);
      gh[0] = ga[63];
    }
#pragma unroll
    for (int c0 = 64; c0 < C::KT; c0 += 16) {
      uint32_t r[16];
      tmem_ld16(tlane + c0, r);
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 16; ++j)
        if (c0 - 63 + j < C::PE_H) gh[c0 - 63 + j] = __uint_as_float(r[j]);
    }
    posenc_bwd<C::H, C::HF>(wp + 3, gh, gx + 3);
  }
}

// d(warped point, hyper coordinates) of one row in f[0, 3 + H) -> the warp / sheet head's pre-activation gradient in f[0, 16)
// (SE3 + sheet: the exp map's in f[0, 16), the sheet head's = d(hyper coordinates) in gh[0, H))
template <class C>
__device__ __forceinline__ void wshead_dy(const BwdParams& p, float* f, float* gh, bool valid, int64_t ray, int64_t gq, int64_t gc,
                                          int lane) {
  if constexpr (C::H == C::G) {
    if (p.mflags & MF_AXIS) {
      // axis-aligned slicing: the hyper coordinates ARE the GLO vector (models.py:533-534), their gradient
      // goes to the table; the (absent) sheet head receives nothing
      const int64_t id = __ldg(p.ids + ray);
      glo_grad_add<C::G>(f + 3, valid, id, p.glo_grad, lane);
#pragma unroll
      for (int i = 0; i < C::G; ++i) f[3 + i] = 0.f;
    }
  }
  if constexpr (C::SE3) {
    // d(warped xyz) -> d(w, v) through the exp map; columns 0..2 / 3..5 of the head's pre-activation gradient
    float x[3], wv[6], gy[3];
    if constexpr (C::WS_ACT) {
#pragma unroll
      for (int i = 0; i < C::H; ++i) gh[i] = f[3 + i];
    }
#pragma unroll
    for (int i = 0; i < 3; ++i) { x[i] = __ldg(p.points + gq * 3 + i); gy[i] = f[i]; }
#pragma unroll
    for (int i = 0; i < 6; ++i) wv[i] = __ldg(p.aux + gc * 6 + i);
    se3_apply_bwd(x, wv, wv + 3, gy, f, f + 3);
  }
}

// the head's dY (f, 16 columns) -> ACT[0, 16) and the dY stash at `chunk`; SE3 + sheet: the sheet head's dY (gh) -> the stash
// at chunk + 2 (SlabMap::d_sheethead) and ACT[16, 32), where the head^T layer leaves it unread (BE_LINSHEET re-writes it)
template <class C>
__device__ __forceinline__ void store_head_dy(const float* f, const float* gh, uint8_t* act_row, uint4* save_row, int chunk) {
  store_features<16>(f, act_row, save_row, chunk);
  if constexpr (C::WS_ACT) {
    float fs[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) fs[i] = i < C::H ? gh[i] : 0.f;
    store_features<16>(fs, act_row + 2 * kChunkBytes, save_row, chunk + 2);
  }
}

// ======================================================================================================
// backward-data
// ======================================================================================================
template <class C>
__global__ void __launch_bounds__(kMlpThreads, 1) mlp_dgrad_kernel(const __grid_constant__ BwdParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  using SM = SmemBwd<C>;
  using Ring = RingStateT<SM::STAGES>;
  constexpr bool PP = true;   // sub-tiles out of phase (see Sched)
  uint8_t* act = smem + SM::ACT;
  uint8_t* inb = smem + SM::INB;
  uint8_t* ring = smem + SM::RING;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + SM::BARS);
  uint64_t* empty = full + SM::STAGES;
  uint64_t* acc_full = empty + SM::STAGES;    // [2]: one per chain
  uint64_t* act_ready = acc_full + 2;         // [2]
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(smem + SM::TMEMP);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int i = 0; i < SM::STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    // one arrival per epilogue warp of the chain
    for (int i = 0; i < 2; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&act_ready[i], 4 * Sched<PP>::SUBS * kEpiSplit); }
    fence_barrier_init();
  }
  if (warp == kIssuerWarp) { tmem_alloc(tmem_ptr, 256 * kSubTiles); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  const Program& prog = p.prog;

  if (warp >= kEpiWarps) {
    setmaxnreg_dec<kRegsFeeder>();
    if (warp == kProducerWarp && lane == 0) {
      Ring rs;
      long long tw = 0;
      for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) produce_tile<PP>(prog, p.weights, ring, full, empty, rs, tw);
      if (p.dbg) p.dbg[blockIdx.x * 8 + 0] = tw;
    } else if (warp == kIssuerWarp) {  // whole warp, converged: see elect_one_sync()
      Ring rs;
      uint32_t ph_ready = 0;
      long long t_ready = 0, t_full = 0;
      const long long t_begin = HN_T0();
      const uint32_t act_s = smem_u32(act), inb_s = smem_u32(inb), ring_s = smem_u32(ring);
      for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
        for (int li = 0; li < prog.nlayers; ++li) {
          for (int chain = 0; chain < Sched<PP>::CHAINS; ++chain) {
            long long t0 = HN_T0();
            mbar_wait(&act_ready[chain], ph_ready);
            t_ready += HN_T0() - t0;
            tc_fence_after();
            issue_layer<PP>(prog, prog.layers[li], chain * Sched<PP>::SUBS, act_s, inb_s, SM::ACT_BYTES, SM::INB_BYTES, ring_s, tmem_base,
                        full, empty, rs, t_full);
            if (elect_one_sync()) umma_commit(&acc_full[chain]);
            __syncwarp();
          }
          ph_ready ^= 1;
        }
      }
      if (p.dbg && lane == 0) {
        p.dbg[blockIdx.x * 8 + 1] = t_ready; p.dbg[blockIdx.x * 8 + 2] = t_full; p.dbg[blockIdx.x * 8 + 3] = HN_T0() - t_begin;
      }
    }
  } else {
    const int sub = warp / (4 * kEpiSplit);
    const int share = (warp >> 2) % kEpiSplit;   // column share of the wide layers; share 0 = the primary warpgroup
    const int quarter = warp & 3;
    auto epilogue = [&](auto primary_tag) {
    constexpr bool PRIMARY = decltype(primary_tag)::value;   // primary: per-row work (heads, chain rules) + its column share
    const int row = quarter * 32 + lane;
    const uint32_t tlane = tmem_base + ((uint32_t)(quarter * 32) << 16) + sub * 256;
    uint8_t* act_row = act + sub * SM::ACT_BYTES + row * 16;
    uint8_t* inb_row = inb + sub * SM::INB_BYTES + row * 16;
    const int chain = PP ? sub : 0;
    uint64_t* my_acc = &acc_full[chain];
    uint64_t* my_ready = &act_ready[chain];
    uint32_t ph_acc = 0;
    long long t_acc = 0, t_pro = 0;
    const long long t_begin = HN_T0();
    for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
      const long long t_tile = HN_T0();
      const int64_t g = (int64_t)tile * kCtaRows + sub * kTileRows + row;
      const bool valid = g < p.n;
      const int64_t gc = valid ? g : p.n - 1;
      const int64_t ray = gc / p.S;
      const int64_t gq = p.pos != nullptr ? ray * p.S_full + __ldg(p.pos + gc) : gc;   // row in the (B, S_full) tensors
      const size_t half = (size_t)tile * (2 * kSubTiles) + sub * 2 + (row >> 6);
      const uint32_t* gate_row = p.gates + half * (size_t)p.g_total * kHalfRows + (row & 63);
      uint4* save_row = reinterpret_cast<uint4*>(p.dsaved + half * (size_t)p.d_total * kHalfChunkBytes) + (row & 63);
      float gh_keep[C::WS_ACT ? C::H : 1] = {};   // SE3 + sheet: the sheet head's dY, from the head's dY to BE_LINSHEET

      if constexpr (PRIMARY && !C::STATIC && !C::NOWARP) {
        if (prog.flags & PF_WARP_ONLY) {
          // warp-stage-only program: dY of the warp / sheet head from the upstream gradient of `warped` (launch rows)
          float f[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) f[i] = 0.f;
          if (valid) {
#pragma unroll
            for (int i = 0; i < C::NWARPED; ++i) f[i] = __ldg(p.g_warped + gc * C::NWARPED + i);
          }
          wshead_dy<C>(p, f, gh_keep, valid, ray, gq, gc, lane);
          store_head_dy<C>(f, gh_keep, act_row, save_row, p.d_rgbhead);
        }
      }
      // prologue: dY of the rgb head = g_rgb * y (1 - y) (Sigmoid, models.py:164)
      if (PRIMARY && !(prog.flags & PF_WARP_ONLY)) {
        float f[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) f[i] = 0.f;
        if (valid) {
#pragma unroll
          for (int i = 0; i < 3; ++i) {
            float y = __ldg(p.rgb + gq * 3 + i);
            f[i] = __ldg(p.g_rgb + gq * 3 + i) * y * (1.f - y);
          }
        }
        store_features<16>(f, act_row, save_row, p.d_rgbhead);
        if constexpr (C::STATIC) {
          // dY of the sigma head: sigma = relu(raw + noise) (rendering.py:150) -> gate on the stored sigma; kept in INB
          // as the A operand of the sigma^T op that accumulates onto final^T, and stashed for the weight gradient
#pragma unroll
          for (int i = 0; i < 16; ++i) f[i] = 0.f;
          if (valid && __ldg(p.sigma + gq) > 0.f) f[0] = __ldg(p.g_sigma + gq);
          store_features<16>(f, inb_row, save_row, p.d_sigma);
        }
      }
      fence_proxy_async_smem();
      tc_fence_before();
      warp_arrive(my_ready);
      t_pro += HN_T0() - t_tile;

      float gx_skip[C::STATIC ? 1 : C::NWARPED] = {};   // skip-layer part of d(warped point, hyper coordinates)
      for (int li = 0; li < prog.nlayers; ++li) {
        const Layer& L = prog.layers[li];
        if (L.epi == BE_MASK) {
          if (L.n_out == kTrunkW) bwd_masked_share<kTrunkW>(share, tlane, gate_row, L.gate_word, act_row, save_row, L.save_chunk, my_acc, ph_acc, t_acc);
          else if (L.n_out == kWsW) bwd_masked_share<kWsW>(share, tlane, gate_row, L.gate_word, act_row, save_row, L.save_chunk, my_acc, ph_acc, t_acc);
          else bwd_masked_share<kRgbW>(share, tlane, gate_row, L.gate_word, act_row, save_row, L.save_chunk, my_acc, ph_acc, t_acc);
          fence_proxy_async_smem();
          if (li + 1 < prog.nlayers) { tc_fence_before(); warp_arrive(my_ready); }
          continue;
        }
        if (!C::STATIC && L.epi == BE_RGB1) {
          bwd_masked_share<kRgbW>(share, tlane, gate_row, L.gate_word, act_row, save_row, L.save_chunk, my_acc, ph_acc, t_acc);
          // alpha column: d softplus(a)/da = sigmoid(a) = 1 - exp(-sigma)
          if constexpr (PRIMARY) {
          float f[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) f[i] = 0.f;
          if (valid) f[0] = __ldg(p.g_sigma + gq) * (-expm1f(-__ldg(p.sigma + gq)));
          store_features<16>(f, act_row + (kRgbW / 8) * kChunkBytes, save_row, L.save_chunk + kRgbW / 8);
          }
          fence_proxy_async_smem(); tc_fence_before(); warp_arrive(my_ready);
          continue;
        }
        { long long t0 = HN_T0(); mbar_wait(my_acc, ph_acc); ph_acc ^= 1; t_acc += HN_T0() - t0; }
        tc_fence_after();
        if (L.epi == BE_LINEAR || L.epi == BE_LINCOND || (C::WS_ACT && L.epi == BE_LINSHEET)) {
          if (L.n_out == kTrunkW) bwd_linear_share<kTrunkW>(share, tlane, act_row, save_row, L.save_chunk);
          else bwd_linear_share<kRgbW>(share, tlane, act_row, save_row, L.save_chunk);
          if constexpr (PRIMARY && C::WS_ACT) {
            if (L.epi == BE_LINSHEET) {   // A operand of the sheet logit^T op of the next layer (kSe3W == kRgbW columns above)
              float fs[16];
#pragma unroll
              for (int i = 0; i < 16; ++i) fs[i] = i < C::H ? gh_keep[i] : 0.f;
              store_features<16>(fs, act_row + (kSe3W / 8) * kChunkBytes, nullptr, 0);
            }
          }
          if constexpr (PRIMARY && !C::STATIC) {
            if (L.epi == BE_LINCOND) {
              // gradient of the GLO condition columns of the view vector (alpha / rgb conditioning, modules.py:283,292),
              // parked in accumulator columns [128, 144) -> gradient of the condition table
              uint32_t r[16];
              tmem_ld16(tlane + kRgbW, r);
              tmem_ld_wait();
              float v[C::G];
#pragma unroll
              for (int i = 0; i < C::G; ++i) v[i] = __uint_as_float(r[i]);
              const int64_t id = __ldg(p.ids + ray);
              HN_CHECK_ID(id, p.n_embed);
              glo_grad_add<C::G>(v, valid, id, p.glo_grad, lane);
            }
          }
        } else if constexpr (PRIMARY && !C::STATIC) {   // (the static program only has BE_MASK / BE_LINEAR layers)
        if (L.epi == BE_SKIPSTORE || L.epi == BE_TRUNKIN) {
          // d(trunk input features) arrives twice: from the skip layer and from layer 0.  The chain rule through the
          // positional encoding is linear in it, so each part is pulled back to d(warped point, hyper coordinates)
          // straight from the fp32 accumulator and the two vectors are added: nothing is parked in shared memory.
          float wp[C::NWARPED], gx[C::NWARPED];
          // trunk-only program: `warped` is warped_in, in launch order; otherwise the level's warped_points output
          const int64_t gw = p.g_warped_out != nullptr ? gc : gq;
#pragma unroll
          for (int i = 0; i < C::NWARPED; ++i) wp[i] = __ldg(p.warped + gw * C::NWARPED + i);
          trunk_in_bwd<C>(tlane, wp, gx);
          if (L.epi == BE_SKIPSTORE) {
#pragma unroll
            for (int i = 0; i < C::NWARPED; ++i) gx_skip[i] = gx[i];
          } else if (p.g_warped_out != nullptr) {
            // trunk-only program: this is the last layer; the gradient goes back to whoever produced warped_in
            if (valid) {
#pragma unroll
              for (int i = 0; i < C::NWARPED; ++i) {
                float v = gx[i] + gx_skip[i];
                // the given point is also an entry of the level's warped_points output: its upstream gradient passes through
                if (p.g_warped != nullptr) v += __ldg(p.g_warped + gq * C::NWARPED + i);
                p.g_warped_out[g * C::NWARPED + i] = v;
              }
            }
          } else if constexpr (!C::NOWARP) {
          float f[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) f[i] = 0.f;
          if (valid) {
#pragma unroll
            for (int i = 0; i < C::NWARPED; ++i) {
              f[i] = gx[i] + gx_skip[i];
              if (p.g_warped != nullptr) f[i] += __ldg(p.g_warped + gq * C::NWARPED + i);
            }
          }
          wshead_dy<C>(p, f, gh_keep, valid, ray, gq, gc, lane);
          store_head_dy<C>(f, gh_keep, act_row, save_row, L.save_chunk);
          }
        } else if constexpr (!C::NOWARP) {  // BE_GLO: d(GLO embedding) of this sample -> per-ray reduction -> atomics on the table gradient
          uint32_t r[16];
          tmem_ld16(tlane + kWsW, r);
          tmem_ld_wait();
          float v[C::G];
#pragma unroll
          for (int i = 0; i < C::G; ++i) v[i] = __uint_as_float(r[i]);
          const int64_t id = __ldg(p.ids + ray);
          HN_CHECK_ID(id, p.n_embed);
          glo_grad_add<C::G>(v, valid, id, p.glo_grad, lane);
        }
        }
        if (li + 1 < prog.nlayers) {
          fence_proxy_async_smem();
          tc_fence_before();
          warp_arrive(my_ready);
        }
      }
    }
    if (p.dbg && threadIdx.x == 0) {
      const long long tt = HN_T0() - t_begin;
      p.dbg[blockIdx.x * 8 + 4] = t_acc; p.dbg[blockIdx.x * 8 + 5] = tt - t_acc - t_pro;
      p.dbg[blockIdx.x * 8 + 6] = t_pro; p.dbg[blockIdx.x * 8 + 7] = tt;
    }
    };   // epilogue
    if (kEpiSplit == 1 || share == 0) { setmaxnreg_inc<kRegsPrimary>(); epilogue(std::true_type{}); }
    else { setmaxnreg_dec<kRegsSecondary>(); epilogue(std::false_type{}); }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kIssuerWarp) tmem_dealloc(tmem_base, 256 * kSubTiles);
}

#ifndef HN_MLP_FWD_VARIANT   // the split-epilogue copy holds the inference forward kernels only
// ======================================================================================================
// weight gradient: for every job, D[N_j, K_j] += dY^T X over this CTA's half tiles (UMMA with both operands
// MN-major straight out of the stash layout), bias gradient by column sums on the CUDA cores.
// ======================================================================================================
constexpr int kWgStages = 3;
constexpr int kWgStageA = 256 * kHalfChunkBytes / 8;  // 32 KB: up to 256 dY columns x 64 rows
constexpr int kWgStageBytes = 2 * kWgStageA;          // + up to 256 X columns
struct WgSmem {
  static constexpr int STAGES = 0;
  static constexpr int BARS = kWgStages * kWgStageBytes;  // full[3], empty[3], acc_full, acc_empty
  static constexpr int TMEMP = BARS + (2 * kWgStages + 2) * 8;
  static constexpr int TOTAL = TMEMP + 16;
};
// Job groups: CTAs of group g run only the jobs with WgradJob::group == g, over 1/(CTAs per group) of the half tiles
// each.  Jobs are spread over the groups by their operand bytes per half tile (the kernel is HBM-bound), largest first.
// 8 groups for the ~30-job tables of the hyper model (measured at 0.5 / 1 / 2 M samples per launch: 8 groups beat 4 by
// 5 / 2.5 / 3 %, 12 and 16 lose to load imbalance) and 4 for the short tables (static NeRF: 12 jobs, 4 groups 502 k against
// 497 k rays/s with 8).
static int wgrad_groups(int njobs) { return njobs >= 24 ? 8 : 4; }
// Spreads the jobs over the groups (largest first) and the grid's CTAs over the groups: every CTA of a group streams the
// group's bytes over 1 / (its CTAs) of the half tiles, so the CTA counts follow the groups' bytes (each next CTA goes to the
// group with the most bytes per CTA).  Round-robin CTA assignment left the heaviest group 6 % above the mean at 8 groups
// (146 chunks on 18 CTAs against 134 on 19); this way it is 3 %.
static void assign_wgrad_groups(WgradTable& t, int groups, int grid, int16_t* group_start) {
  int order[kMaxJobs];
  int64_t load[16] = {};
  auto cost = [&](int i) { return (int)t.jobs[i].dy_nchunks + t.jobs[i].x0_nchunks + t.jobs[i].x1_nchunks; };
  for (int i = 0; i < t.njobs; ++i) order[i] = i;
  std::stable_sort(order, order + t.njobs, [&](int a, int b) { return cost(a) > cost(b); });
  for (int k = 0; k < t.njobs; ++k) {
    int best = 0;
    for (int g = 1; g < groups; ++g) if (load[g] < load[best]) best = g;
    t.jobs[order[k]].group = (uint8_t)best;
    load[best] += cost(order[k]);
  }
  int ctas[16];
  for (int g = 0; g < groups; ++g) ctas[g] = 1;
  for (int c = groups; c < grid; ++c) {
    int best = 0;
    for (int g = 1; g < groups; ++g)
      if (load[g] * ctas[best] > load[best] * ctas[g]) best = g;
    ++ctas[best];
  }
  group_start[0] = 0;
  for (int g = 0; g < groups; ++g) group_start[g + 1] = (int16_t)(group_start[g] + ctas[g]);
}

// Positional-encoding window w_k(alpha) = 0.5 (1 - cos(pi clamp(alpha - k, 0, 1))) of encoded column e (PackBlock::win_c):
// exactly 1 for alpha >= k + 1 (cospif(1) = -1), exactly 0 for alpha <= k.
__device__ __forceinline__ float pe_window(float alpha, uint8_t win_c, int e) {
  const int C = win_c & ~kWinIdentity;
  if (win_c & kWinIdentity) {
    if (e < C) return 1.f;
    e -= C;
  }
  const float x = fminf(fmaxf(alpha - (float)(e / (2 * C)), 0.f), 1.f);
  return 0.5f * (1.f - cospif(x));
}

struct WgradParams {
  WgradTable tab;
  const uint8_t* saved; const uint8_t* dsaved;
  const float* pe_alpha;   // windowed tables (mlp_wgrad_kernel<true>): device {warp, sheet, nerf, hyper} alphas
  float* flat_grad;
  int64_t n_half;
  int x_total, d_total;
  int groups;   // job groups (WgradJob::group < groups)
  int16_t group_start[17];   // CTAs [group_start[g], group_start[g + 1]) serve group g (share of the grid ~ the group's bytes)
};

// WIN: the X stash holds the unwindowed encodings, so the accumulator holds dY^T pe; a flush segment with a window
// scales it by w on its way out (dW of W diag(w) = (dY^T pe) diag(w)).
template <bool WIN>
__global__ void __launch_bounds__(192, 1) mlp_wgrad_kernel(const __grid_constant__ WgradParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + WgSmem::BARS);
  uint64_t* empty = full + kWgStages;
  uint64_t* acc_full = empty + kWgStages;
  uint64_t* acc_empty = acc_full + 1;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(smem + WgSmem::TMEMP);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int i = 0; i < kWgStages; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1 + 4); }
    mbar_init(acc_full, 1);
    mbar_init(acc_empty, 128);
    fence_barrier_init();
  }
  if (warp == 1) { tmem_alloc(tmem_ptr, 512); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  // CTA b belongs to the job group whose CTA range holds b and owns a contiguous range of half tiles inside it.  Every CTA flushes its
  // partial dW of the jobs it ran with fp32 atomics; with one group that is the whole 5.9 MB gradient per CTA (876 MB of
  // atomic traffic and ~0.56 ms per launch, measured); with G groups each CTA runs 1/G of the jobs over G times more
  // half tiles, the operand traffic is unchanged and the flush traffic drops G-fold.
  int my_group = 0;
  while (my_group + 1 < p.groups && (int)blockIdx.x >= p.group_start[my_group + 1]) ++my_group;
  const int ctas_in_group = p.group_start[my_group + 1] - p.group_start[my_group];
  const int64_t per = (p.n_half + ctas_in_group - 1) / ctas_in_group;
  const int64_t h0 = (int64_t)((int)blockIdx.x - p.group_start[my_group]) * per;
  const int64_t h1 = min(h0 + per, p.n_half);
  const int njobs = p.tab.njobs;

  if (warp == 0) {
    if (lane == 0 && h0 < h1) {
      int slot = 0; uint32_t phase = 0;
      for (int ji = 0; ji < njobs; ++ji) {
        const WgradJob& J = p.tab.jobs[ji];
        if (J.group != my_group) continue;
        const uint32_t a_bytes = J.dy_nchunks * kHalfChunkBytes;
        const uint32_t b0_bytes = J.x0_nchunks * kHalfChunkBytes, b1_bytes = J.x1_nchunks * kHalfChunkBytes;
        for (int64_t h = h0; h < h1; ++h) {
          uint8_t* st = smem + slot * kWgStageBytes;
          mbar_wait(&empty[slot], phase ^ 1);
          mbar_arrive_expect_tx(&full[slot], a_bytes + b0_bytes + b1_bytes);
          bulk_g2s(st, p.dsaved + ((size_t)h * p.d_total + J.dy_chunk) * kHalfChunkBytes, a_bytes, &full[slot]);
          bulk_g2s(st + kWgStageA, p.saved + ((size_t)h * p.x_total + J.x0_chunk) * kHalfChunkBytes, b0_bytes, &full[slot]);
          if (b1_bytes)
            bulk_g2s(st + kWgStageA + b0_bytes, p.saved + ((size_t)h * p.x_total + J.x1_chunk) * kHalfChunkBytes, b1_bytes,
                       &full[slot]);
          if (++slot == kWgStages) { slot = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (h0 < h1) {  // whole warp, converged
      int slot = 0; uint32_t phase = 0, ph_empty = 0;
      // both operands MN-major straight out of the stash layout: 8 columns contiguous (16 B), K = rows (16 B stride);
      // LBO = 8 rows (128 B), SBO = one chunk (kHalfChunkBytes)
      constexpr uint32_t kHi = (1u << 14) | (kHalfChunkBytes >> 4);
      const uint32_t st0 = smem_u32(smem);
      bool first = true;
      for (int ji = 0; ji < njobs; ++ji) {
        const WgradJob& J = p.tab.jobs[ji];
        if (J.group != my_group) continue;
        const uint32_t ncols = (J.x0_nchunks + J.x1_nchunks) * 8;  // UMMA N
        const uint32_t idesc = make_idesc_bf16(128, ncols, 1, 1);
        const bool two = J.mblocks == 2;
        const uint32_t d1 = tmem_base + ncols;
        if (!first) { mbar_wait(acc_empty, ph_empty); ph_empty ^= 1; tc_fence_after(); }
        first = false;
        for (int64_t h = h0; h < h1; ++h) {
          mbar_wait(&full[slot], phase);
          tc_fence_after();
          if (elect_one_sync()) {
            const uint32_t a_lo = ((st0 + slot * kWgStageBytes) >> 4) | ((128u >> 4) << 16);
            const uint32_t b_lo = a_lo + (kWgStageA >> 4);
            uint32_t acc = h > h0;
#pragma unroll
            for (int ks = 0; ks < kHalfRows / 16; ++ks) {
              const uint64_t bd = ((uint64_t)kHi << 32) | (b_lo + ks * 16);
              umma_bf16(tmem_base, ((uint64_t)kHi << 32) | (a_lo + ks * 16), bd, idesc, acc);
              if (two) umma_bf16(d1, ((uint64_t)kHi << 32) | (a_lo + ks * 16 + ((16 * kHalfChunkBytes) >> 4)), bd, idesc, acc);
              acc = 1;
            }
            umma_commit(&empty[slot]);
          }
          __syncwarp();
          if (++slot == kWgStages) { slot = 0; phase ^= 1; }
        }
        if (elect_one_sync()) umma_commit(acc_full);
        __syncwarp();
      }
    }
  } else if (h0 < h1) {
    // warps 2..5: bias column sums while streaming, TMEM flush at the end of every job
    const int quarter = warp & 3;
    const int wr = warp - 2;  // 0..3: which quarter of the dY chunks this warp reduces
    const uint32_t tlane = tmem_base + ((uint32_t)(quarter * 32) << 16);
    int slot = 0; uint32_t phase = 0, ph_acc = 0;
    for (int ji = 0; ji < njobs; ++ji) {
      const WgradJob& J = p.tab.jobs[ji];
      if (J.group != my_group) continue;
      const int ncols = (J.x0_nchunks + J.x1_nchunks) * 8;
      // chunks [c_lo, c_hi) of the dY part belong to this warp (<= 8 chunks)
      const int cpw = (J.dy_nchunks + 3) / 4;
      const int c_lo = min(wr * cpw, (int)J.dy_nchunks), c_hi = min(c_lo + cpw, (int)J.dy_nchunks);
      float bs[8][8];
#pragma unroll
      for (int a = 0; a < 8; ++a)
#pragma unroll
        for (int b = 0; b < 8; ++b) bs[a][b] = 0.f;
      for (int64_t h = h0; h < h1; ++h) {
        mbar_wait(&full[slot], phase);
        if (J.nbias) {
          const uint8_t* st = smem + slot * kWgStageBytes;
#pragma unroll
          for (int a = 0; a < 8; ++a) {
            if (c_lo + a < c_hi) {
#pragma unroll
              for (int rr = 0; rr < kHalfRows; rr += 32) {
                uint4 v = *reinterpret_cast<const uint4*>(st + (c_lo + a) * kHalfChunkBytes + (rr + lane) * 16);
                bs[a][0] += bf16_lo(v.x); bs[a][1] += bf16_hi(v.x); bs[a][2] += bf16_lo(v.y); bs[a][3] += bf16_hi(v.y);
                bs[a][4] += bf16_lo(v.z); bs[a][5] += bf16_hi(v.z); bs[a][6] += bf16_lo(v.w); bs[a][7] += bf16_hi(v.w);
              }
            }
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[slot]);
        if (++slot == kWgStages) { slot = 0; phase ^= 1; }
      }
      // bias gradient: reduce over the 32 lanes (rows), one atomic per column
      if (J.nbias) {
#pragma unroll
        for (int a = 0; a < 8; ++a) {
          if (c_lo + a < c_hi) {
#pragma unroll
            for (int b = 0; b < 8; ++b) {
              float v = bs[a][b];
#pragma unroll
              for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
              const int col = (c_lo + a) * 8 + b;
              if (lane == 0) {
                for (int s = 0; s < J.nbias; ++s) {
                  const BiasSeg& B = J.bias[s];
                  if (col >= B.col0 && col < B.col0 + B.ncols) atomicAdd(p.flat_grad + B.dst + (col - B.col0), v);
                }
              }
            }
          }
        }
      }
      // flush the accumulator
      mbar_wait(acc_full, ph_acc); ph_acc ^= 1;
      tc_fence_after();
      for (int mb = 0; mb < J.mblocks; ++mb) {
        const int drow = mb * 128 + quarter * 32 + lane;  // row in dY-column space
        for (int c0 = 0; c0 < ncols; c0 += 16) {
          uint32_t r[16];
          tmem_ld16(tlane + mb * ncols + c0, r);
          tmem_ld_wait();
          for (int s = 0; s < J.nflush; ++s) {
            const FlushSeg& F = J.flush[s];
            if (drow >= F.row0 && drow < F.row0 + F.nrows) {
              // this thread's 16 accumulator columns are 16 consecutive floats of one dW row: four 16-byte vector
              // reductions when the row is 16-byte aligned (ld % 4 == 0, the wide layers), scalar ones otherwise
              float* dst = p.flat_grad + F.dst + (int64_t)(drow - F.row0) * F.ld + (c0 - (int)F.col0);
              const bool vec = (reinterpret_cast<uintptr_t>(dst) & 15) == 0;
              uint32_t v[16];
#pragma unroll
              for (int j = 0; j < 16; ++j) v[j] = r[j];
              if (WIN && F.win != kNoWin) {   // columns outside [col0, col0 + ncols) get a weight too but are not written
                const float a = p.pe_alpha[F.win - 1];
#pragma unroll
                for (int j = 0; j < 16; ++j)
                  v[j] = __float_as_uint(__uint_as_float(r[j]) * pe_window(a, F.win_c, (int)F.win_e0 + c0 + j - (int)F.col0));
              }
#pragma unroll
              for (int j = 0; j < 16; j += 4) {
                const int col = c0 + j;
                if (vec && col >= F.col0 && col + 4 <= F.col0 + F.ncols) {
                  red_add_v4(dst + j, v[j], v[j + 1], v[j + 2], v[j + 3]);
                } else {
#pragma unroll
                  for (int jj = j; jj < j + 4; ++jj)
                    if (c0 + jj >= F.col0 && c0 + jj < F.col0 + F.ncols) atomicAdd(dst + jj, __uint_as_float(v[jj]));
                }
              }
            }
          }
        }
      }
      tc_fence_before();
      mbar_arrive(acc_empty);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// ======================================================================================================
// weight packing
// ======================================================================================================
struct PackParams {
  PackTable tab;
  const float* flat;
  const float* pe_alpha;   // device {warp, sheet, nerf, hyper} alphas of the windowed tables; NULL: no window
  uint8_t* blob;
  int64_t bias_off, glo_off;
  int64_t glo_src;
  int glo_floats;
};

__global__ void pack_kernel(const __grid_constant__ PackParams p) {
  const int oi = blockIdx.y;
  if (oi < p.tab.nops) {
    const PackOp& op = p.tab.ops[oi];
    const int npk = op.n * (op.k / 8);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < npk; i += gridDim.x * blockDim.x) {
      const int chunk = i / op.n, n = i % op.n;
      float v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = 0.f;
      for (int b = op.blk0; b < op.blk0 + op.nblk; ++b) {
        const PackBlock& B = p.tab.blocks[b];
        if (n < B.n0 || n >= B.n0 + B.nn) continue;
        // windowed block: W diag(w) in fp32, rounded to bf16 below; the source column runs along k in the forward
        // images (sk == 1) and along n in the transposed ones
        const float a = p.pe_alpha != nullptr && B.win != kNoWin ? __ldg(p.pe_alpha + B.win - 1) : 0.f;
        const bool win = p.pe_alpha != nullptr && B.win != kNoWin;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          int k = chunk * 8 + j;
          if (k >= B.k0 && k < B.k0 + B.kk) {
            if (B.sk == kBiasPairStride) {   // folded bias: bf16(b), bf16(b - bf16(b))
              const float bv = __ldg(p.flat + B.src + (int64_t)(n - B.n0) * B.sn);
              const float hi = __uint_as_float(pack_bf16(bv, 0.f) << 16);
              v[j] = k == B.k0 ? hi : bv - hi;
            } else {
              v[j] = __ldg(p.flat + B.src + (int64_t)(n - B.n0) * B.sn + (int64_t)(k - B.k0) * B.sk);
              if (win) v[j] *= pe_window(a, B.win_c, (int)B.win_e0 + (B.sk == 1 ? k - B.k0 : n - B.n0));
            }
          }
        }
      }
      uint4 o;
      o.x = pack_bf16(v[0], v[1]); o.y = pack_bf16(v[2], v[3]); o.z = pack_bf16(v[4], v[5]); o.w = pack_bf16(v[6], v[7]);
      reinterpret_cast<uint4*>(p.blob + (size_t)op.w_off16 * 16)[i] = o;
    }
  } else {
    // biases + GLO table copy
    float* bias = reinterpret_cast<float*>(p.blob + p.bias_off);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < p.tab.bias_floats; i += gridDim.x * blockDim.x) {
      float v = 0.f;
      for (int b = 0; b < p.tab.nbias; ++b) {
        const BiasBlock& B = p.tab.bias[b];
        if (i >= B.dst && i < B.dst + B.cnt) v = __ldg(p.flat + B.src + (i - B.dst));
      }
      bias[i] = v;
    }
    float* glo = reinterpret_cast<float*>(p.blob + p.glo_off);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < p.glo_floats; i += gridDim.x * blockDim.x)
      glo[i] = __ldg(p.flat + p.glo_src + i);
  }
}

#endif  // !HN_MLP_FWD_VARIANT

// ------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------
static unsigned long long* g_dbg = nullptr;
static int64_t tiles_of(int64_t n) { return (n + kCtaRows - 1) / kCtaRows; }   // CTA tiles (256 rows)

template <class K, class P>
static cudaError_t launch_mlp(K kernel, int grid, int smem, cudaStream_t stream, const P& params) {
  kernel<<<grid, kMlpThreads, smem, stream>>>(params);
  return cudaGetLastError();
}

// cudaFuncAttributeMaxDynamicSharedMemorySize is set once per (kernel, device) instead of before every launch
template <class K>
static int set_smem(K kernel, int bytes, const char* what) {
  static thread_local std::unordered_map<const void*, int> done;   // kernel -> device it was set on
  int dev = 0;
  if (cudaError_t e = cudaGetDevice(&dev)) return set_cuda_error(e, what);
  auto it = done.find((const void*)kernel);
  if (it != done.end() && it->second == dev) return 0;
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess) done[(const void*)kernel] = dev;
  return set_cuda_error(e, what);
}

// The layer programs / slab maps depend on the descriptor only, the pack and weight-gradient tables additionally on
// (level, parameter offsets): both are cached per thread, so a launch does not rebuild several KB of tables.
struct PlanCache {
  bool have_plan = false, have_tables = false, windowed = false;
  hn_model_desc desc;
  int level = -1;
  int64_t offs[HN_NUM_PARAM_TENSORS];
  ModelPlan plan;
};
static ModelPlan& cached_plan(const hn_model_desc& d, int level = -1, const int64_t* offsets = nullptr,
                              bool windowed = false) {
  static thread_local PlanCache c;
  if (!c.have_plan || memcmp(&c.desc, &d, sizeof(d)) != 0) {
    build_plan(d, &c.plan);
    c.desc = d; c.have_plan = true; c.have_tables = false;
  }
  if (offsets != nullptr) {
    const size_t nb = sizeof(int64_t) * c.plan.info.n_params;
    if (!c.have_tables || c.level != level || c.windowed != windowed || memcmp(c.offs, offsets, nb) != 0) {
      build_tables(d, level, offsets, windowed, &c.plan);
      memcpy(c.offs, offsets, nb);
      c.level = level; c.windowed = windowed; c.have_tables = true;
    }
  }
  return c.plan;
}

}  // namespace hn

using namespace hn;

#ifndef HN_MLP_FWD_VARIANT
extern "C" int hn_query(const hn_model_desc* desc, int64_t n_samples, hn_sizes* out) {
  if (!desc || !out) return set_error(-2, "hn_query: null pointer");
  if (int rc = validate_desc(*desc)) return rc;
  if (n_samples < 0) return set_error(-1, "hn_query: negative n_samples");
  const ModelPlan& plan = cached_plan(*desc);
  memset(out, 0, sizeof(*out));
  const int64_t halves = 2 * kSubTiles * tiles_of(n_samples);
  out->packed_bytes = plan.layout.total;
  // X slabs, then the ReLU gate words ([half tile][g_total][64 rows] uint32)
  out->saved_bytes = halves * plan.info.x_total * kHalfChunkBytes + halves * plan.info.g_total * kHalfRows * 4;
  out->workspace_bytes = halves * plan.info.d_total * kHalfChunkBytes;
  // the warp-stage-only launches (hn_mlp_fwd_warp / hn_mlp_bwd_warp_*) stash the slab-map prefixes alone
  out->warp_saved_bytes = halves * plan.info.x_warp * kHalfChunkBytes + halves * plan.info.g_warp * kHalfRows * 4;
  out->warp_workspace_bytes = halves * plan.info.d_warp * kHalfChunkBytes;
  const Dims& m = plan.dims;
  auto lin = [](int64_t out_f, int64_t in_f) { return out_f * in_f + out_f; };
  if (is_static(*desc)) {   // NeRF(D=8, W=256): 595 844 parameters at the default 63 / 27 input channels
    out->flat_param_floats = lin(kTrunkW, m.pe_x) + 6 * lin(kTrunkW, kTrunkW) + lin(kTrunkW, kTrunkW + m.pe_x) + lin(1, kTrunkW) +
                             lin(kTrunkW, kTrunkW) + lin(kRgbW, kTrunkW + m.pe_v) + lin(3, kRgbW);
    return 0;
  }
  // parameters of the canonical slots this configuration has (include/hypernerf_b200.h)
  int64_t cnt = plan.info.glo_floats;
  if (m.se3) {
    cnt += lin(kSe3W, m.in_w) + 4 * lin(kSe3W, kSe3W) + lin(kSe3W, kSe3W + m.in_w) + lin(kSe3W, kSe3W) +
           2 * (lin(kSe3W, kSe3W) + lin(3, kSe3W));
  } else if (!m.nowarp) {
    cnt += lin(kWarpW, m.in_w) + 4 * lin(kWarpW, kWarpW) + lin(kWarpW, kWarpW + m.in_w) + lin(3, kWarpW);
  }
  if (!m.nowarp && !m.axis)   // the HyperSheetMLP of bendy-sheet slicing, with either warp field
    cnt += lin(kSheetW, m.in_s) + 4 * lin(kSheetW, kSheetW) + lin(kSheetW, kSheetW + m.in_s) + lin(m.H, kSheetW);
  int64_t lvl = lin(kTrunkW, m.in_t) + 7 * lin(kTrunkW, kTrunkW) + lin(kTrunkW, kTrunkW + m.in_t) + lin(kRgbW, kTrunkW) +
                lin(kRgbW, kRgbW + m.pe_v + (m.cond_r ? m.G : 0)) + 3 * lin(kRgbW, kRgbW) + lin(3, kRgbW) +
                lin(1, kRgbW + (m.cond_a ? m.G : 0));
  out->flat_param_floats = cnt + 2 * lvl;
  return 0;
}

static int pack_impl(const hn_model_desc* desc, const float* flat_params, const int64_t* param_offsets, int level,
                     void* packed, const float* pe_alpha, void* stream) {
  if (!desc || !flat_params || !param_offsets || !packed) return set_error(-2, "hn_pack_weights: null pointer");
  if (level < 0 || level > 1) return set_error(-1, "hn_pack_weights: level must be 0 or 1");
  if (int rc = validate_desc(*desc)) return rc;
  const ModelPlan& plan = cached_plan(*desc, level, param_offsets, pe_alpha != nullptr);
  PackParams pp;
  pp.tab = plan.pack;
  pp.flat = flat_params;
  pp.pe_alpha = pe_alpha;
  pp.blob = (uint8_t*)packed;
  pp.bias_off = plan.layout.bias_off;
  pp.glo_off = plan.layout.glo_off;
  pp.glo_src = plan.info.glo_param >= 0 ? param_offsets[plan.info.glo_param] : 0;
  if (plan.info.glo_param >= 0 && pp.glo_src < 0) return set_error(-2, "hn_pack_weights: the GLO table of this configuration has no offset");
  pp.glo_floats = plan.info.glo_floats;
  dim3 grid(16, plan.pack.nops + 1);
  pack_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(pp);
  return set_cuda_error(cudaGetLastError(), "hn_pack_weights");
}

extern "C" int hn_pack_weights(const hn_model_desc* desc, const float* flat_params, const int64_t* param_offsets, int level,
                               void* packed, void* stream) {
  return pack_impl(desc, flat_params, param_offsets, level, packed, nullptr, stream);
}

extern "C" int hn_pack_weights_windowed(const hn_model_desc* desc, const float* flat_params, const int64_t* param_offsets,
                                        int level, void* packed, const float* pe_alpha, void* stream) {
  if (!pe_alpha) return set_error(-2, "hn_pack_weights_windowed: null pe_alpha");
  if (desc && is_static(*desc)) return set_error(-13, "hn_pack_weights_windowed: the static NeRF has no encoding window");
  return pack_impl(desc, flat_params, param_offsets, level, packed, pe_alpha, stream);
}

#endif  // !HN_MLP_FWD_VARIANT

// run-time model flags of the fused kernels
static int model_flags(const hn_model_desc& d) {
  int f = 0;
  if (d.flags & HN_FLAG_SLICE_AXIS) f |= MF_AXIS;
  if (d.flags & (HN_FLAG_ALPHA_COND | HN_FLAG_RGB_COND)) f |= MF_COND;
  return f;
}
// which compile-time shape serves a descriptor: 0 static, 1 hyper_dim 2, 2 hyper_dim 4, 3 hyper_dim 8, 4 no warp, 5 SE3 warp
// + axis-aligned slicing, 6 SE3 warp + bendy sheet
static int shape_of(const hn_model_desc& d) {
  if (is_static(d)) return 0;
  if (d.flags & HN_FLAG_WARP_SE3) return (d.flags & HN_FLAG_SLICE_AXIS) ? 5 : 6;
  if (!has_warp(d)) return 4;
  return d.hyper_dim == 2 ? 1 : d.hyper_dim == 4 ? 2 : 3;
}
#define HN_DISPATCH_SHAPE(shape, MACRO) \
  switch (shape) {                      \
    case 0: MACRO(CfgStatic); break;    \
    case 1: MACRO(Cfg1); break;         \
    case 2: MACRO(CfgH4); break;        \
    case 3: MACRO(CfgH8); break;        \
    case 5: MACRO(CfgSE3); break;       \
    case 6: MACRO(CfgSE3S); break;      \
    default: MACRO(CfgT); break;        \
  }

template <class C, bool STASH>
static int launch_fwd(const FwdParams& fp, int grid, void* stream) {
  if (int rc = set_smem(mlp_fwd_kernel<C, STASH>, Smem<C>::TOTAL, "hn_mlp_fwd: smem attr")) return rc;
  return set_cuda_error(launch_mlp(mlp_fwd_kernel<C, STASH>, grid, Smem<C>::TOTAL, (cudaStream_t)stream, fp), "hn_mlp_fwd");
}

// warped_in != NULL: trunk-only program (hn_mlp_fwd_trunk; always the case for a model without warp: warped_in = points)
static int mlp_fwd_impl(const hn_model_desc* desc, const void* packed, const float* points, const float* warped_in,
                        const float* viewdirs, const int64_t* ids, const float* noise, float noise_std, int64_t B, int S,
                        const int32_t* pos, int S_full, float* sigma, float* rgb, float* warped, void* saved, float* aux,
                        void* stream) {
  if (!desc || !packed || (!points && !warped_in) || !viewdirs || !sigma || !rgb) return set_error(-2, "hn_mlp_fwd: null pointer");
  if (B < 0 || S <= 0) return set_error(-1, "hn_mlp_fwd: bad B/S");
  if (pos != nullptr && S_full < S) return set_error(-1, "hn_mlp_fwd: scattered rows need S_full >= S");
  if (int rc = validate_desc(*desc)) return rc;
  const bool stat = is_static(*desc);
  const int mflags = stat ? 0 : model_flags(*desc);
  if (!stat && !has_warp(*desc) && !warped_in) { warped_in = points; warped = nullptr; }
  const bool trunk = warped_in != nullptr;
  if (!stat && (desc->flags & HN_FLAG_WARP_SE3) && !trunk && saved != nullptr && !aux)
    return set_error(-2, "hn_mlp_fwd: the SE3 warp needs the aux buffer when the stash is written");
  if (trunk && stat) return set_error(-13, "hn_mlp_fwd_trunk: the static model has no warp / sheet stage to skip");
  if (!stat && !ids && (!trunk || (mflags & MF_COND))) return set_error(-2, "hn_mlp_fwd: null ids");
  if (B == 0) return 0;
  const ModelPlan& plan = cached_plan(*desc);
  FwdParams fp;
  // the stash-writing forward runs the programs without bias K steps and adds the biases in its epilogue
  const bool train = saved != nullptr;
  fp.prog = trunk ? (train ? plan.fwd_trunk_train : plan.fwd_trunk) : (train ? plan.fwd_train : plan.fwd);
  fp.warped_in = warped_in;
  fp.weights = (const uint8_t*)packed + plan.layout.fwd_off;
  fp.bias = (const float*)((const uint8_t*)packed + plan.layout.bias_off);
  fp.glo = (const float*)((const uint8_t*)packed + plan.layout.glo_off);
  fp.points = points; fp.viewdirs = viewdirs; fp.ids = ids; fp.noise = noise; fp.noise_std = noise_std;
  fp.n = B * S; fp.S = S; fp.n_embed = desc->num_embeddings;
  fp.view_freqs = desc->view_freqs; fp.mflags = mflags;
  fp.pos = pos; fp.S_full = pos != nullptr ? S_full : S;
  int64_t nt = tiles_of(fp.n);
  if (nt > 0x7fffffff) return set_error(-1, "hn_mlp_fwd: too many samples");
  fp.n_tiles = (int)nt;
  fp.x_total = plan.info.x_total;
  fp.x_in_ws = plan.info.x_in0; fp.x_in_t = plan.info.x_in_t; fp.x_in_v = plan.info.x_in_v;
  fp.sigma = sigma; fp.rgb = rgb; fp.warped = warped; fp.saved = (uint8_t*)saved;
  fp.aux = saved != nullptr ? aux : nullptr;
  fp.g_total = plan.info.g_total;
  fp.gates = saved ? (uint32_t*)((uint8_t*)saved + (size_t)(2 * kSubTiles) * nt * plan.info.x_total * kHalfChunkBytes) : nullptr;
  fp.dbg = g_dbg;
  const int grid = (int)std::min<int64_t>(nt, num_sms());
#ifdef HN_MLP_FWD_VARIANT   // the split-epilogue copy serves the launches without a stash only
#define HN_LAUNCH_FWD(CFG) return launch_fwd<CFG, false>(fp, grid, stream)
#else
#define HN_LAUNCH_FWD(CFG) return train ? launch_fwd<CFG, true>(fp, grid, stream) : launch_fwd<CFG, false>(fp, grid, stream)
#endif
  HN_DISPATCH_SHAPE(shape_of(*desc), HN_LAUNCH_FWD)
#undef HN_LAUNCH_FWD
  return set_error(-1, "hn_mlp_fwd: unreachable");
}

#if defined(HN_MLP_FV_LINKED) && !defined(HN_MLP_FWD_VARIANT)
extern "C" int hn_mlp_fwd_fv(const hn_model_desc*, const void*, const float*, const float*, const int64_t*, const float*, float,
                             int64_t, int, const int32_t*, int, float*, float*, float*, void*, float*, void*);
extern "C" int hn_mlp_fwd_trunk_fv(const hn_model_desc*, const void*, const float*, const float*, const int64_t*, const float*,
                                   float, int64_t, int, const int32_t*, int, float*, float*, float*, void*, void*);
// every launch without a stash runs on the split-epilogue copy (hn_mlp_fv.o)
#define HN_MLP_FV_CALL(fn, ...) if (saved == nullptr) return fn(__VA_ARGS__)
#else
#define HN_MLP_FV_CALL(fn, ...)
#endif

extern "C" HN_FV_HIDDEN int hn_mlp_fwd(const hn_model_desc* desc, const void* packed, const float* points, const float* viewdirs,
                          const int64_t* ids, const float* noise, float noise_std, int64_t B, int S, const int32_t* pos,
                          int S_full, float* sigma, float* rgb, float* warped, void* saved, float* aux, void* stream) {
  HN_MLP_FV_CALL(hn_mlp_fwd_fv, desc, packed, points, viewdirs, ids, noise, noise_std, B, S, pos, S_full, sigma, rgb, warped,
                      saved, aux, stream);
  if (!points) return set_error(-2, "hn_mlp_fwd: null pointer");
  return mlp_fwd_impl(desc, packed, points, nullptr, viewdirs, ids, noise, noise_std, B, S, pos, S_full, sigma, rgb, warped,
                      saved, aux, stream);
}

extern "C" HN_FV_HIDDEN int hn_mlp_fwd_trunk(const hn_model_desc* desc, const void* packed, const float* warped_in, const float* viewdirs,
                                const int64_t* ids, const float* noise, float noise_std, int64_t B, int S, const int32_t* pos,
                                int S_full, float* sigma, float* rgb, float* warped, void* saved, void* stream) {
  HN_MLP_FV_CALL(hn_mlp_fwd_trunk_fv, desc, packed, warped_in, viewdirs, ids, noise, noise_std, B, S, pos, S_full, sigma, rgb,
                      warped, saved, stream);
  if (!warped_in) return set_error(-2, "hn_mlp_fwd_trunk: null pointer");
  return mlp_fwd_impl(desc, packed, nullptr, warped_in, viewdirs, ids, noise, noise_std, B, S, pos, S_full, sigma, rgb, warped,
                      saved, nullptr, stream);
}

#if defined(HN_MLP_FV_LINKED) && !defined(HN_MLP_FWD_VARIANT)
extern "C" int hn_mlp_fwd_warp_fv(const hn_model_desc*, const void*, const float*, const int64_t*, int64_t, int, float*, void*,
                                  float*, void*);
#endif

// checks shared by the warp-stage-only entry points: a hyper model with a warp stage, a positive sample count
static int check_warp_only(const hn_model_desc* desc, int64_t B, int S, const char* what) {
  if (is_static(*desc)) return set_error(-13, (std::string(what) + ": the static NeRF has no warp stage").c_str());
  if (!has_warp(*desc)) return set_error(-13, (std::string(what) + ": this model has no warp field (use_warp=False)").c_str());
  if (B <= 0 || S <= 0) return set_error(-1, (std::string(what) + ": B and S must be positive").c_str());
  return validate_desc(*desc);
}

extern "C" HN_FV_HIDDEN int hn_mlp_fwd_warp(const hn_model_desc* desc, const void* packed, const float* points, const int64_t* ids,
                                            int64_t B, int S, float* warped, void* saved, float* aux, void* stream) {
  HN_MLP_FV_CALL(hn_mlp_fwd_warp_fv, desc, packed, points, ids, B, S, warped, saved, aux, stream);
  if (!desc || !packed || !points || !ids || !warped) return set_error(-2, "hn_mlp_fwd_warp: null pointer");
  if (int rc = check_warp_only(desc, B, S, "hn_mlp_fwd_warp")) return rc;
  if ((desc->flags & HN_FLAG_WARP_SE3) && saved != nullptr && !aux)
    return set_error(-2, "hn_mlp_fwd_warp: the SE3 warp needs the aux buffer when the stash is written");
  const ModelPlan& plan = cached_plan(*desc);
  const bool train = saved != nullptr;
  FwdParams fp;
  memset(&fp, 0, sizeof(fp));
  fp.prog = train ? plan.fwd_warp_train : plan.fwd_warp;
  fp.weights = (const uint8_t*)packed + plan.layout.fwd_off;
  fp.bias = (const float*)((const uint8_t*)packed + plan.layout.bias_off);
  fp.glo = (const float*)((const uint8_t*)packed + plan.layout.glo_off);
  fp.points = points; fp.ids = ids;
  fp.n = B * S; fp.S = S; fp.n_embed = desc->num_embeddings;
  fp.view_freqs = desc->view_freqs; fp.mflags = model_flags(*desc);
  fp.S_full = S;
  const int64_t nt = tiles_of(fp.n);
  if (nt > 0x7fffffff) return set_error(-1, "hn_mlp_fwd_warp: too many samples");
  fp.n_tiles = (int)nt;
  // the warp-only stash: slab-map prefixes as the per-half-tile strides (PlanInfo::x_warp / g_warp)
  fp.x_total = plan.info.x_warp;
  fp.x_in_ws = plan.info.x_in0; fp.x_in_t = kNone; fp.x_in_v = kNone;
  fp.warped = warped; fp.saved = (uint8_t*)saved; fp.aux = aux;
  fp.g_total = plan.info.g_warp;
  fp.gates = train ? (uint32_t*)((uint8_t*)saved + (size_t)(2 * kSubTiles) * nt * plan.info.x_warp * kHalfChunkBytes) : nullptr;
  fp.dbg = g_dbg;
  const int grid = (int)std::min<int64_t>(nt, num_sms());
#ifdef HN_MLP_FWD_VARIANT
#define HN_LAUNCH_FWD(CFG) return launch_fwd<CFG, false>(fp, grid, stream)
#else
#define HN_LAUNCH_FWD(CFG) return train ? launch_fwd<CFG, true>(fp, grid, stream) : launch_fwd<CFG, false>(fp, grid, stream)
#endif
  HN_DISPATCH_SHAPE(shape_of(*desc), HN_LAUNCH_FWD)
#undef HN_LAUNCH_FWD
  return set_error(-1, "hn_mlp_fwd_warp: unreachable");
}

#ifndef HN_MLP_FWD_VARIANT
template <class C>
static int launch_fwd_tangent(const FwdParams& fp, int grid, void* stream) {
  if (int rc = set_smem(mlp_fwd_kernel<C, true, true>, Smem<C>::TOTAL, "hn_mlp_fwd_warp_tangent: smem attr")) return rc;
  return set_cuda_error(launch_mlp(mlp_fwd_kernel<C, true, true>, grid, Smem<C>::TOTAL, (cudaStream_t)stream, fp),
                        "hn_mlp_fwd_warp_tangent");
}

// Jacobian of the translation warp (ModelPlan::fwd_warp_tangent): one launch of 3 x the primal's tiles, gated by the gate
// words of the primal's warp-only stash (hn_mlp_fwd_warp with a stash); tangent_saved (3 x hn_sizes.warp_saved_bytes,
// nullable) receives the tangents' X slabs for hn_mlp_bwd_warp_weights.
extern "C" int hn_mlp_fwd_warp_tangent(const hn_model_desc* desc, const void* packed, const float* points, const void* primal_saved,
                                       int64_t B, int S, float* jac, void* tangent_saved, void* stream) {
  if (!desc || !packed || !points || !primal_saved || !jac) return set_error(-2, "hn_mlp_fwd_warp_tangent: null pointer");
  if (int rc = check_warp_only(desc, B, S, "hn_mlp_fwd_warp_tangent")) return rc;
  if (desc->flags & HN_FLAG_WARP_SE3)
    return set_error(-13, "hn_mlp_fwd_warp_tangent: the Jacobian is built for the translation warp only, not for SE3");
  const ModelPlan& plan = cached_plan(*desc);
  FwdParams fp;
  memset(&fp, 0, sizeof(fp));
  fp.prog = plan.fwd_warp_tangent;
  fp.weights = (const uint8_t*)packed + plan.layout.fwd_off;
  fp.bias = (const float*)((const uint8_t*)packed + plan.layout.bias_off);
  fp.glo = (const float*)((const uint8_t*)packed + plan.layout.glo_off);
  fp.points = points;
  fp.n = B * S; fp.S = S; fp.n_embed = desc->num_embeddings;
  fp.view_freqs = desc->view_freqs; fp.mflags = model_flags(*desc);
  fp.S_full = S;
  const int64_t nt = tiles_of(fp.n);
  if (3 * nt > 0x7fffffff) return set_error(-1, "hn_mlp_fwd_warp_tangent: too many samples");
  fp.n_tiles = (int)(3 * nt);
  fp.x_total = plan.info.x_warp;
  fp.x_in_ws = plan.info.x_in0; fp.x_in_t = kNone; fp.x_in_v = kNone;
  fp.saved = (uint8_t*)tangent_saved;
  fp.g_total = plan.info.g_warp;
  fp.gates = (uint32_t*)((uint8_t*)primal_saved + (size_t)(2 * kSubTiles) * nt * plan.info.x_warp * kHalfChunkBytes);
  fp.jac = jac;
  fp.dbg = g_dbg;
  const int grid = (int)std::min<int64_t>(3 * nt, num_sms());
  switch (shape_of(*desc)) {
    case 1: return launch_fwd_tangent<Cfg1>(fp, grid, stream);
    case 2: return launch_fwd_tangent<CfgH4>(fp, grid, stream);
    case 3: return launch_fwd_tangent<CfgH8>(fp, grid, stream);
    default: return set_error(-13, "hn_mlp_fwd_warp_tangent: no tangent kernel for this configuration");
  }
}

static int mlp_bwd_impl(const hn_model_desc* desc, const void* packed, const int64_t* ids, const float* sigma,
                        const float* rgb, const float* warped, const void* saved, const float* g_sigma, const float* g_rgb,
                        const float* g_warped, int64_t B, int S, const int32_t* pos, int S_full, int level,
                        const int64_t* param_offsets, float* flat_grad, void* workspace, void* stream, bool do_data,
                        bool do_weights, bool trunk = false,
                        float* g_warped_out = nullptr,     // trunk: trunk-only programs (hn_mlp_bwd_trunk*)
                        const float* points = nullptr, const float* aux = nullptr,     // SE3 warp, full program only
                        const float* pe_alpha = nullptr) {   // windowed weight gradient (hn_mlp_bwd_*weights_windowed)
  if (!desc || !saved || !param_offsets || !flat_grad || !workspace) return set_error(-2, "hn_mlp_bwd: null pointer");
  const bool stat = desc && is_static(*desc);
  const bool nowarp = !stat && !has_warp(*desc);
  if (!stat && (desc->flags & HN_FLAG_WARP_SE3) && !trunk && do_data && (!points || !aux))
    return set_error(-2, "hn_mlp_bwd: the SE3 warp needs the sample points and the forward's aux buffer");
  const int mflags = stat ? 0 : model_flags(*desc);
  if (nowarp) trunk = true;   // a model without warp only has the template: `warped` are the raw sample points
  if (trunk && do_data && !g_warped_out && !nowarp) return set_error(-2, "hn_mlp_bwd_trunk: null pointer");
  if (trunk && stat) return set_error(-13, "hn_mlp_bwd_trunk: the static model has no warp / sheet stage to skip");
  if (do_data && (!packed || !sigma || !rgb || !g_sigma || !g_rgb ||
                  (!stat && ((!ids && (!trunk || (mflags & MF_COND))) || !warped))))
    return set_error(-2, "hn_mlp_bwd: null pointer");
  if (B < 0 || S <= 0) return set_error(-1, "hn_mlp_bwd: bad B/S");
  if (level < 0 || level > 1) return set_error(-1, "hn_mlp_bwd: level must be 0 or 1");
  if (int rc = validate_desc(*desc)) return rc;
  if (B == 0) return 0;
  // the data gradient reads no offset-dependent table: only the weight gradient (re)builds them
  const ModelPlan& plan = cached_plan(*desc, level, do_weights ? param_offsets : nullptr, pe_alpha != nullptr);
  const int64_t n = B * S;
  const int64_t nt = tiles_of(n);
  if (nt > 0x7fffffff) return set_error(-1, "hn_mlp_bwd: too many samples");
  if (do_data) {
    BwdParams bp;
    bp.prog = trunk ? plan.bwd_trunk : plan.bwd;
    bp.g_warped_out = g_warped_out;
    bp.weights = (const uint8_t*)packed + plan.layout.bwd_off;
    bp.ids = ids; bp.sigma = sigma; bp.rgb = rgb; bp.warped = warped;
    bp.g_sigma = g_sigma; bp.g_rgb = g_rgb; bp.g_warped = g_warped;
    bp.points = points; bp.aux = aux;
    bp.saved = (const uint8_t*)saved; bp.dsaved = (uint8_t*)workspace;
    bp.g_total = plan.info.g_total;
    bp.gates = (const uint32_t*)((const uint8_t*)saved + (size_t)(2 * kSubTiles) * nt * plan.info.x_total * kHalfChunkBytes);
    bp.glo_grad = nullptr;
    if (plan.info.glo_param >= 0) {
      if (param_offsets[plan.info.glo_param] < 0) return set_error(-2, "hn_mlp_bwd: the GLO table of this configuration has no gradient offset");
      bp.glo_grad = flat_grad + param_offsets[plan.info.glo_param];
    }
    bp.mflags = mflags;
    bp.pos = pos; bp.S_full = pos != nullptr ? S_full : S;
    bp.n = n; bp.S = S; bp.n_embed = desc->num_embeddings;
    bp.n_tiles = (int)nt;
    bp.x_total = plan.info.x_total; bp.d_total = plan.info.d_total;
    bp.d_rgbhead = plan.info.d_rgbhead; bp.d_sigma = plan.info.d_sigma;
    bp.dbg = g_dbg;
    const int grid = (int)std::min<int64_t>(nt, num_sms());
#define HN_LAUNCH_BWD(CFG)                                                                                                  \
  do {                                                                                                                      \
    if (int rc = set_smem(mlp_dgrad_kernel<CFG>, SmemBwd<CFG>::TOTAL, "hn_mlp_bwd: dgrad smem attr")) return rc;            \
    if (int rc = set_cuda_error(launch_mlp(mlp_dgrad_kernel<CFG>, grid, SmemBwd<CFG>::TOTAL, (cudaStream_t)stream, bp),     \
                                "hn_mlp_bwd: dgrad launch")) return rc;                                                     \
  } while (0)
    HN_DISPATCH_SHAPE(shape_of(*desc), HN_LAUNCH_BWD)
#undef HN_LAUNCH_BWD
  }
  if (do_weights) {
    WgradParams wp;
    wp.tab = trunk ? plan.wgrad_trunk : plan.wgrad;
    wp.saved = (const uint8_t*)saved; wp.dsaved = (const uint8_t*)workspace;
    wp.pe_alpha = pe_alpha;
    wp.flat_grad = flat_grad;
    wp.n_half = 2 * kSubTiles * nt;
    wp.x_total = plan.info.x_total; wp.d_total = plan.info.d_total;
    const auto wgrad_kernel = pe_alpha != nullptr ? mlp_wgrad_kernel<true> : mlp_wgrad_kernel<false>;
    if (int rc = set_smem(wgrad_kernel, WgSmem::TOTAL, "hn_mlp_bwd: wgrad smem attr")) return rc;
    const int wgrid = (int)std::min<int64_t>(wp.n_half, num_sms());
    wp.groups = wp.n_half >= 8 * (int64_t)wgrid ? std::min(wgrad_groups(wp.tab.njobs), wgrid) : 1;
    assign_wgrad_groups(wp.tab, wp.groups, wgrid, wp.group_start);
    wgrad_kernel<<<wgrid, 192, WgSmem::TOTAL, (cudaStream_t)stream>>>(wp);
    if (int rc = set_cuda_error(cudaGetLastError(), "hn_mlp_bwd: wgrad launch")) return rc;
  }
  return 0;
}

extern "C" int hn_mlp_bwd(const hn_model_desc* desc, const void* packed, const int64_t* ids, const float* sigma,
                          const float* rgb, const float* warped, const void* saved, const float* g_sigma,
                          const float* g_rgb, const float* g_warped, int64_t B, int S, const int32_t* pos, int S_full, int level,
                          const int64_t* param_offsets, float* flat_grad, void* workspace, const float* points,
                          const float* aux, void* stream) {
  return mlp_bwd_impl(desc, packed, ids, sigma, rgb, warped, saved, g_sigma, g_rgb, g_warped, B, S, pos, S_full, level,
                      param_offsets, flat_grad, workspace, stream, true, true, false, nullptr, points, aux);
}

extern "C" int hn_mlp_bwd_data(const hn_model_desc* desc, const void* packed, const int64_t* ids, const float* sigma,
                               const float* rgb, const float* warped, const void* saved, const float* g_sigma,
                               const float* g_rgb, const float* g_warped, int64_t B, int S, const int32_t* pos, int S_full,
                               int level, const int64_t* param_offsets, float* flat_grad, void* workspace,
                               const float* points, const float* aux, void* stream) {
  return mlp_bwd_impl(desc, packed, ids, sigma, rgb, warped, saved, g_sigma, g_rgb, g_warped, B, S, pos, S_full, level,
                      param_offsets, flat_grad, workspace, stream, true, false, false, nullptr, points, aux);
}

extern "C" int hn_mlp_bwd_weights(const hn_model_desc* desc, const void* saved, int64_t B, int S, int level,
                                  const int64_t* param_offsets, float* flat_grad, const void* workspace, void* stream) {
  return mlp_bwd_impl(desc, nullptr, nullptr, nullptr, nullptr, nullptr, saved, nullptr, nullptr, nullptr, B, S, nullptr, 0,
                      level, param_offsets, flat_grad, (void*)workspace, stream, false, true);
}

extern "C" int hn_mlp_bwd_trunk(const hn_model_desc* desc, const void* packed, const int64_t* ids, const float* sigma,
                                const float* rgb, const float* warped_in, const void* saved, const float* g_sigma,
                                const float* g_rgb, const float* g_warped, int64_t B, int S, const int32_t* pos, int S_full,
                                int level, const int64_t* param_offsets, float* flat_grad, float* g_warped_in, void* workspace,
                                void* stream) {
  return mlp_bwd_impl(desc, packed, ids, sigma, rgb, warped_in, saved, g_sigma, g_rgb, g_warped, B, S, pos, S_full, level,
                      param_offsets, flat_grad, workspace, stream, true, true, true, g_warped_in);
}

extern "C" int hn_mlp_bwd_trunk_data(const hn_model_desc* desc, const void* packed, const int64_t* ids, const float* sigma,
                                     const float* rgb, const float* warped_in, const void* saved, const float* g_sigma,
                                     const float* g_rgb, const float* g_warped, int64_t B, int S, const int32_t* pos,
                                     int S_full, int level, const int64_t* param_offsets, float* flat_grad, float* g_warped_in,
                                     void* workspace, void* stream) {
  return mlp_bwd_impl(desc, packed, ids, sigma, rgb, warped_in, saved, g_sigma, g_rgb, g_warped, B, S, pos, S_full, level,
                      param_offsets, flat_grad, workspace, stream, true, false, true, g_warped_in);
}

extern "C" int hn_mlp_bwd_trunk_weights(const hn_model_desc* desc, const void* saved, int64_t B, int S, int level,
                                        const int64_t* param_offsets, float* flat_grad, const void* workspace, void* stream) {
  return mlp_bwd_impl(desc, nullptr, nullptr, nullptr, nullptr, nullptr, saved, nullptr, nullptr, nullptr, B, S, nullptr, 0,
                      level, param_offsets, flat_grad, (void*)workspace, stream, false, true, true, nullptr);
}

extern "C" int hn_mlp_bwd_weights_windowed(const hn_model_desc* desc, const void* saved, int64_t B, int S, int level,
                                           const int64_t* param_offsets, float* flat_grad, const void* workspace,
                                           const float* pe_alpha, void* stream) {
  if (!pe_alpha) return set_error(-2, "hn_mlp_bwd_weights_windowed: null pe_alpha");
  if (desc && is_static(*desc)) return set_error(-13, "hn_mlp_bwd_weights_windowed: the static NeRF has no encoding window");
  return mlp_bwd_impl(desc, nullptr, nullptr, nullptr, nullptr, nullptr, saved, nullptr, nullptr, nullptr, B, S, nullptr, 0,
                      level, param_offsets, flat_grad, (void*)workspace, stream, false, true, false, nullptr, nullptr, nullptr,
                      pe_alpha);
}

extern "C" int hn_mlp_bwd_trunk_weights_windowed(const hn_model_desc* desc, const void* saved, int64_t B, int S, int level,
                                                 const int64_t* param_offsets, float* flat_grad, const void* workspace,
                                                 const float* pe_alpha, void* stream) {
  if (!pe_alpha) return set_error(-2, "hn_mlp_bwd_trunk_weights_windowed: null pe_alpha");
  if (desc && is_static(*desc))
    return set_error(-13, "hn_mlp_bwd_trunk_weights_windowed: the static NeRF has no encoding window");
  return mlp_bwd_impl(desc, nullptr, nullptr, nullptr, nullptr, nullptr, saved, nullptr, nullptr, nullptr, B, S, nullptr, 0,
                      level, param_offsets, flat_grad, (void*)workspace, stream, false, true, true, nullptr, nullptr, nullptr,
                      pe_alpha);
}

// Warp-stage-only backward (level-0 blob, hn_mlp_fwd_warp's stash): data gradient from g_warped, then / or the weight
// gradient of the warp / sheet jobs.
static int mlp_bwd_warp_impl(const hn_model_desc* desc, const void* packed, const int64_t* ids, const void* saved,
                             const float* g_warped, int64_t B, int S, const int64_t* param_offsets, float* flat_grad,
                             void* workspace, const float* points, const float* aux, const float* pe_alpha, bool do_data,
                             bool do_weights, void* stream, const char* what) {
  if (!desc || !saved || !param_offsets || !flat_grad || !workspace) return set_error(-2, (std::string(what) + ": null pointer").c_str());
  if (do_data && (!packed || !ids || !g_warped)) return set_error(-2, (std::string(what) + ": null pointer").c_str());
  if (int rc = check_warp_only(desc, B, S, what)) return rc;
  if (do_data && (desc->flags & HN_FLAG_WARP_SE3) && (!points || !aux))
    return set_error(-2, (std::string(what) + ": the SE3 warp needs the sample points and the forward's aux buffer").c_str());
  const ModelPlan& plan = cached_plan(*desc, 0, do_weights ? param_offsets : nullptr, pe_alpha != nullptr);
  const int64_t n = B * S;
  const int64_t nt = tiles_of(n);
  if (nt > 0x7fffffff) return set_error(-1, (std::string(what) + ": too many samples").c_str());
  if (do_data) {
    BwdParams bp;
    memset(&bp, 0, sizeof(bp));
    bp.prog = plan.bwd_warp;
    bp.weights = (const uint8_t*)packed + plan.layout.bwd_off;
    bp.ids = ids; bp.g_warped = g_warped;
    bp.points = points; bp.aux = aux;
    bp.saved = (const uint8_t*)saved; bp.dsaved = (uint8_t*)workspace;
    bp.g_total = plan.info.g_warp;
    bp.gates = (const uint32_t*)((const uint8_t*)saved + (size_t)(2 * kSubTiles) * nt * plan.info.x_warp * kHalfChunkBytes);
    if (param_offsets[plan.info.glo_param] < 0) return set_error(-2, (std::string(what) + ": the GLO table has no gradient offset").c_str());
    bp.glo_grad = flat_grad + param_offsets[plan.info.glo_param];
    bp.mflags = model_flags(*desc);
    bp.S_full = S;
    bp.n = n; bp.S = S; bp.n_embed = desc->num_embeddings;
    bp.n_tiles = (int)nt;
    bp.x_total = plan.info.x_warp; bp.d_total = plan.info.d_warp;
    bp.d_rgbhead = plan.slabs.d_wshead;   // the dY slab the PF_WARP_ONLY prologue writes
    bp.d_sigma = kNone;
    bp.dbg = g_dbg;
    const int grid = (int)std::min<int64_t>(nt, num_sms());
#define HN_LAUNCH_BWD(CFG)                                                                                                  \
  do {                                                                                                                      \
    if (int rc = set_smem(mlp_dgrad_kernel<CFG>, SmemBwd<CFG>::TOTAL, what)) return rc;                                     \
    if (int rc = set_cuda_error(launch_mlp(mlp_dgrad_kernel<CFG>, grid, SmemBwd<CFG>::TOTAL, (cudaStream_t)stream, bp), what)) \
      return rc;                                                                                                            \
  } while (0)
    HN_DISPATCH_SHAPE(shape_of(*desc), HN_LAUNCH_BWD)
#undef HN_LAUNCH_BWD
  }
  if (do_weights) {
    WgradParams wp;
    wp.tab = plan.wgrad_warp;
    wp.saved = (const uint8_t*)saved; wp.dsaved = (const uint8_t*)workspace;
    wp.pe_alpha = pe_alpha;
    wp.flat_grad = flat_grad;
    wp.n_half = 2 * kSubTiles * nt;
    wp.x_total = plan.info.x_warp; wp.d_total = plan.info.d_warp;
    const auto wgrad_kernel = pe_alpha != nullptr ? mlp_wgrad_kernel<true> : mlp_wgrad_kernel<false>;
    if (int rc = set_smem(wgrad_kernel, WgSmem::TOTAL, what)) return rc;
    const int wgrid = (int)std::min<int64_t>(wp.n_half, num_sms());
    wp.groups = wp.n_half >= 8 * (int64_t)wgrid ? std::min(wgrad_groups(wp.tab.njobs), wgrid) : 1;
    assign_wgrad_groups(wp.tab, wp.groups, wgrid, wp.group_start);
    wgrad_kernel<<<wgrid, 192, WgSmem::TOTAL, (cudaStream_t)stream>>>(wp);
    if (int rc = set_cuda_error(cudaGetLastError(), what)) return rc;
  }
  return 0;
}

extern "C" int hn_mlp_bwd_warp_data(const hn_model_desc* desc, const void* packed, const int64_t* ids, const void* saved,
                                    const float* g_warped, int64_t B, int S, const int64_t* grad_offsets, float* flat_grad,
                                    void* workspace, const float* points, const float* aux, void* stream) {
  return mlp_bwd_warp_impl(desc, packed, ids, saved, g_warped, B, S, grad_offsets, flat_grad, workspace, points, aux, nullptr,
                           true, false, stream, "hn_mlp_bwd_warp_data");
}

extern "C" int hn_mlp_bwd_warp_weights(const hn_model_desc* desc, const void* saved, int64_t B, int S,
                                       const int64_t* grad_offsets, float* flat_grad, const void* workspace,
                                       const float* pe_alpha, void* stream) {
  return mlp_bwd_warp_impl(desc, nullptr, nullptr, saved, nullptr, B, S, grad_offsets, flat_grad, (void*)workspace, nullptr,
                           nullptr, pe_alpha, false, true, stream, "hn_mlp_bwd_warp_weights");
}

#if HN_ROLE_TIMING
// profiling hook of the role-timing builds (include/hypernerf_b200_probe.h; not part of the drop-in surface): device buffer
// of 8 x uint64 per CTA that the fused kernels fill with per-role cycle counters; NULL switches it off.
extern "C" int hn_debug_set_timing_buffer(void* dev_buffer) {
  g_dbg = (unsigned long long*)dev_buffer;
  return 0;
}
#endif
#endif  // !HN_MLP_FWD_VARIANT
