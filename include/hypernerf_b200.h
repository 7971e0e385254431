/* hypernerf_b200 — C-ABI of the B200-native HyperNeRF per-ray hot path.
 *
 * This is the drop-in boundary B2 of SURVEY.md §8(b): the reference (songrise/HyperNeRF-torch) has no FFI
 * of its own — its hot path is Python calling stock torch ops — so each entry point below replaces one
 * Python function of the reference, cited as file:line into the reference tree.  The Python shim in
 * hypernerf_torch_b200/ (same class / function names and signatures as the reference) is the only caller.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; every pointer is a DEVICE pointer unless stated otherwise.
 *   - every function returns int: 0 = ok, <0 = argument / shape error, >0 = cudaError_t of the launch.
 *     hn_last_error() returns a thread-local message for the last non-zero return.
 *   - nothing allocates, synchronises or throws; all buffers are caller-owned; kernels are enqueued on the
 *     cudaStream_t passed as `void* stream`.
 *   - all float tensors are fp32 row-major contiguous; ids are int64.
 */
#ifndef HYPERNERF_B200_H
#define HYPERNERF_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define HN_ABI_VERSION 4

/* Topology of one NerfModel (reference: hypernerf/models.py:111-309): NerfMLP (modules.py:172-298) with trunk 8x256
 * skip@4 and rgb branch 4x128, optionally conditioned on a GLO embedding, behind one of the working combinations of
 * SURVEY.md App. B.2:
 *   warp + bendy_sheet     TranslationField 6x128 skip@4 (warping.py:28-125) + HyperSheetMLP 6x64 skip@4 (modules.py:302-337)
 *   warp + axis_aligned    TranslationField + hyper point = the GLO vector itself (models.py:533-534; hyper_dim == glo_dim)
 *   no warp + no slicing   the template alone on the raw sample points (models.py:545-581 with use_warp=False)
 * Instantiated shapes: glo_dim 8, hyper_dim 1..8 (0 without warp), xyz / hyper freqs 10 / 6, view freqs <= 6,
 * warp / sheet freqs 10 / 7.  Anything else is rejected by hn_query with a message (there is no fallback). */
typedef struct hn_model_desc {
  int32_t glo_dim;        /* G: GLO embedding width (opt.py:99)                                  */
  int32_t hyper_dim;      /* H: hyper_slice_out_dim (opt.py:92)                                  */
  int32_t xyz_freqs;      /* template xyz posenc_orig freqs (opt.py:110)                         */
  int32_t hyper_freqs;    /* template hyper posenc_orig freqs (opt.py:112)                       */
  int32_t view_freqs;     /* viewdir posenc_orig freqs (opt.py:114)                              */
  int32_t warp_freqs;     /* TranslationField.n_freq, hard-coded 10 (warping.py:74)              */
  int32_t sheet_freqs;    /* HyperSheetMLP.n_freq, hard-coded 7 (modules.py:313)                 */
  int32_t num_embeddings; /* rows of warp_embed.embed.weight (train.py:42-46 -> 100)             */
  int32_t flags;          /* HN_FLAG_*                                                           */
  int32_t reserved[7];
} hn_model_desc;

#define HN_FLAG_WARP_TRANSLATION 1  /* use_warp with TranslationField                            */
#define HN_FLAG_SLICE_BENDY 2       /* hyper_slice_method == 'bendy_sheet'                       */
#define HN_FLAG_SLICE_AXIS 8        /* hyper_slice_method == 'axis_aligned_plane': hyper point = GLO vector (models.py:533-534) */
#define HN_FLAG_ALPHA_COND 16       /* use_nerf_embed + use_alpha_cond: alpha head input [bottleneck | GLO] (modules.py:283)   */
#define HN_FLAG_RGB_COND 32         /* use_nerf_embed + use_rgb_cond: rgb branch input [bottleneck | view PE | GLO] (:292)     */
#define HN_FLAG_WARP_SE3 64         /* SE3Field warp (warping.py:128-272, rigid_body.py:55-83) instead of TranslationField; set
                                       together with HN_FLAG_WARP_TRANSLATION's place taken: flags = WARP_SE3 | SLICE_AXIS
                                       (config 5: glo_dim = hyper_dim = 8) or WARP_SE3 | SLICE_BENDY (SE3Field + HyperSheetMLP,
                                       HyperNeRF's "DS" model: glo_dim 8, hyper_dim 2, sheet_freqs 7; other hyper_dim are
                                       rejected by hn_query with a message); warp_freqs = 8 either way.  The
                                       reference never instantiates SE3Field and its exp map is not runnable batched
                                       (SURVEY.md App. B.1): parity for this flag is against the batched restatement in oracle/ */
#define HN_FLAG_STATIC_NERF 4       /* static baseline models/nerf.py:41-123 (one NeRF per blob; xyz_freqs 10,
                                       view_freqs 4; glo/hyper/warp/sheet fields ignored).  hn_mlp_fwd then returns
                                       sigma = relu(raw + noise * noise_std) (rendering.py:150) and rgb; ids / warped
                                       may be NULL; `level` is ignored.  Canonical parameter order = state_dict order
                                       of NeRF: xyz_encoding_{1..8}.0.{weight,bias}, xyz_encoding_final.{weight,bias},
                                       dir_encoding.0.{weight,bias}, sigma.{weight,bias}, rgb.0.{weight,bias}          */
#define HN_NUM_STATIC_PARAM_TENSORS 24

/* Canonical parameter order = state_dict order of the reference model (SURVEY.md App. A.6):
 *   0                      warp_embed.embed.weight (E,G)
 *   1..14                  hyper_sheet_mlp.mlp.linears.{0..5}.{weight,bias}, logit_layer.{weight,bias}
 *   15..28                 warp_field.mlp.linears.{0..5}.{weight,bias}, logit_layer.{weight,bias}
 *   29 + 32*level + ...    nerf_mlps_{coarse,fine}: trunk linears 0..7 + logit (18), bottleneck (2),
 *                          rgb linears 0..3 + logit (10), alpha (2)
 *   93                     nerf_embed.embed.weight (E,G): the condition table when there is no warp (models.py:425-430;
 *                          with a warp the condition is warp_embed, slot 0, models.py:421-423)
 *   94..101                SE3Field only: w_net.linears.0, w_net.logit_layer, v_net.linears.0, v_net.logit_layer
 *                          {weight,bias}; its trunk (linears 0..5 + logit_layer) takes slots 15..28
 * Offsets tables give the element offset of tensor i relative to a base pointer; the tensors need not be
 * contiguous with each other (the Python shim passes base = lowest parameter address).  A tensor the configuration
 * does not have (sheet MLP with axis-aligned slicing, warp MLP without warp, ...) has a NEGATIVE offset. */
#define HN_NUM_PARAM_TENSORS 102

typedef struct hn_sizes {
  int64_t packed_bytes;       /* one level's packed bf16 weights (forward + transposed) + fp32 biases */
  int64_t saved_bytes;        /* activations saved by hn_mlp_fwd for n_samples (training)           */
  int64_t workspace_bytes;    /* hn_mlp_bwd scratch (pre-activation gradients) for n_samples        */
  int64_t flat_param_floats;  /* total parameter count                                              */
  int64_t warp_saved_bytes;   /* activations saved by hn_mlp_fwd_warp for n_samples (0 without warp) */
  int64_t warp_workspace_bytes; /* hn_mlp_bwd_warp_* scratch for n_samples (0 without warp)          */
  int64_t reserved[2];
} hn_sizes;

int hn_abi_version(void);
const char* hn_last_error(void);

/* Buffer sizes for a model and a sample count (n_samples = rays * samples-per-ray of one level). */
int hn_query(const hn_model_desc* desc, int64_t n_samples, hn_sizes* out /* host */);

/* fp32 master parameters -> kernel-layout bf16 blobs of one level (0 = coarse, 1 = fine).
 * Replaces nothing in the reference (nn.Linear holds (out,in) fp32); it is the per-step re-layout.
 * param_offsets: HOST array of HN_NUM_PARAM_TENSORS element offsets. */
int hn_pack_weights(const hn_model_desc* desc, const float* flat_params, const int64_t* param_offsets /* host */,
                    int level, void* packed, void* stream);

/* model_utils.sample_along_rays (model_utils.py:6-41).  lower/upper: (Nc,) stratum bounds computed by the
 * caller with the reference's own torch ops (bit-exact linspace); u: (B,Nc) uniform draws or NULL
 * (non-stratified: z = lower).  Writes z (B,Nc) and points (B,Nc,3) = o + z*d. */
int hn_sample_coarse(const float* origins, const float* dirs, const float* u, const float* lower,
                     const float* upper, int64_t B, int Nc, float* z, float* points, void* stream);

/* model_utils.piecewise_constant_pdf + sample_pdf (model_utils.py:160-232).
 *   bins    (B, nb+1) contiguous, or NULL: computed in-kernel as .5*(z[1:]+z[:-1]) of z_coarse (the
 *           z_vals_mid of models.py:752; requires nb == Nc-2)
 *   weights row b starts at weights + b*w_stride and has nb entries (models.py:753 passes the strided view
 *           coarse_weights[..., 1:-1]: pointer w+1, stride Nc)
 *   u       (B,Nf) uniform draws (the caller materialises linspace for the non-stratified case)
 * Writes sorted z_fine (B,Nc+Nf) = sort(cat[z_coarse, samples]), points (B,Nc+Nf,3) (nullable), optional
 * bin_idx (B,Nf) int32 = searchsorted(cdf,u,right=True). */
int hn_sample_pdf(const float* z_coarse, const float* bins, const float* weights, int64_t w_stride, const float* u,
                  const float* origins, const float* dirs, int64_t B, int Nc, int nb, int Nf, float* z_fine,
                  float* points, int32_t* bin_idx, void* stream);
/* The same, additionally reporting where the merge put every input: pos_coarse (B,Nc) / pos_new (B,Nf) int32 = index in
 * the sorted output row of coarse depth i / of the i-th smallest new sample (a permutation of 0..Nc+Nf-1 per ray).  The
 * drop-in model uses it to evaluate inherited and new depths in separate launches (hn_mlp_fwd_trunk).  pos_coarse[i]
 * refers to input element i only for ascending z_coarse rows — what sample_along_rays produces; a non-ascending row is
 * sorted first and i then counts in ascending order. */
int hn_sample_pdf_ranks(const float* z_coarse, const float* bins, const float* weights, int64_t w_stride, const float* u,
                        const float* origins, const float* dirs, int64_t B, int Nc, int nb, int Nf, float* z_fine,
                        float* points, int32_t* bin_idx, int32_t* pos_coarse, int32_t* pos_new, void* stream);

/* model_utils.volumetric_rendering + compute_depth_index (model_utils.py:43-107, 319-362).
 * flags: HN_COMP_*.  eps = 1e-5 and last_delta = 1e7 reproduce the HyperNeRF path; the static
 * models/rendering.py:137-172 path uses 1e-10 / 1e10 and HN_COMP_ACC_ALL. */
#define HN_COMP_WHITE_BKGD 1
#define HN_COMP_ACC_ALL 2 /* acc sums every weight (no sample at infinity) */
int hn_composite_fwd(const float* sigma, const float* rgb, const float* z, const float* dirs, int64_t B, int S,
                     int flags, float eps, float last_delta, float* out_rgb, float* depth, float* med_depth,
                     float* acc, float* weights, int64_t* med_idx, void* stream);
/* Reverse of the above: gradients w.r.t. sigma (B,S) and rgb samples (B,S,3).  g_depth / g_acc / g_weights
 * may be NULL. */
int hn_composite_bwd(const float* sigma, const float* rgb, const float* z, const float* dirs, int64_t B, int S,
                     int flags, float eps, float last_delta, const float* g_out_rgb, const float* g_depth,
                     const float* g_acc, const float* g_weights, float* g_sigma, float* g_rgb, void* stream);

/* filter_sigma (models.py:35-63; applied to the fine level only, models.py:768): out[i] = values[i] where sigma[i] >=
 * dust_threshold (if use_dust) and points[i] lies inside bbox = {xmin, xmax, ymin, ymax, zmin, zmax} (HOST pointer, NULL =
 * no box test), else 0.  Forward: values = sigma.  Backward: values = the upstream gradient (same mask).  n = B * S. */
int hn_filter_sigma(const float* points, const float* sigma, const float* values, int64_t n, float dust_threshold, int use_dust,
                    const float* bbox_host, float* out, void* stream);

/* render_samples up to and including query_template (models.py:587-650 -> :447-493): GLO lookup, posenc_orig,
 * TranslationField, HyperSheetMLP, NerfMLP, noise_regularize, Softplus — one fused tcgen05 kernel.
 * points (B,S,3); viewdirs (B,3) (the reference passes the raw ray directions, models.py:717-720);
 * ids: (B,) int64 row of metadata['time']; noise: (B,S) standard-normal draws or NULL; noise_std scales it.
 * Outputs sigma (B,S) post-softplus, rgb (B,S,3) post-sigmoid, warped (B,S,3+H);
 * saved: activation stash for hn_mlp_bwd (NULL = inference).
 * Scattered rows (pos != NULL): the launch evaluates S of the S_full samples of every ray — launch row j of ray b is
 * sample pos[b*S + j] (int32) of that ray: points / noise are read and sigma / rgb / warped written at that position of
 * (B,S_full,...) tensors.  The drop-in model evaluates the fine level's new and inherited depths in two launches that
 * fill one sorted (B,Nc+Nf) row (models.py:752-767).  pos == NULL: S_full is ignored, rows are the launch rows.
 * aux: SE3 warp only, training only: (B,S,6) fp32 scratch that receives the screw parameters (w, v) of every launch row for
 * the backward pass; NULL otherwise. */
int hn_mlp_fwd(const hn_model_desc* desc, const void* packed, const float* points, const float* viewdirs,
               const int64_t* ids, const float* noise, float noise_std, int64_t B, int S, const int32_t* pos, int S_full,
               float* sigma, float* rgb, float* warped, void* saved, float* aux, void* stream);

/* autograd of hn_mlp_fwd: accumulates parameter gradients of `level` (and the shared warp / sheet / GLO
 * gradients) into flat_grad (fp32); grad_offsets: HOST array of HN_NUM_PARAM_TENSORS element offsets into
 * flat_grad.  g_warped may be NULL.  workspace: hn_sizes.workspace_bytes of scratch.  pos / S_full as in the forward
 * (sigma, rgb, warped, g_sigma, g_rgb, g_warped are the (B,S_full,...) tensors).  points / aux: SE3 warp only (the sample
 * points the forward saw and the (w, v) it wrote), NULL otherwise. */
int hn_mlp_bwd(const hn_model_desc* desc, const void* packed, const int64_t* ids, const float* sigma, const float* rgb,
               const float* warped, const void* saved, const float* g_sigma, const float* g_rgb, const float* g_warped,
               int64_t B, int S, const int32_t* pos, int S_full, int level, const int64_t* grad_offsets /* host */,
               float* flat_grad, void* workspace, const float* points, const float* aux, void* stream);

/* The two halves of hn_mlp_bwd, separately callable (hn_mlp_bwd == data then weights on the same stream):
 *   hn_mlp_bwd_data     back-propagates through every layer (tcgen05, transposed weights), writes the
 *                       pre-activation gradients to `workspace` and accumulates the GLO-table gradient;
 *   hn_mlp_bwd_weights  dW = dY^T X and db = sum dY over all samples from `saved` + `workspace`. */
int hn_mlp_bwd_data(const hn_model_desc* desc, const void* packed, const int64_t* ids, const float* sigma,
                    const float* rgb, const float* warped, const void* saved, const float* g_sigma, const float* g_rgb,
                    const float* g_warped, int64_t B, int S, const int32_t* pos, int S_full, int level,
                    const int64_t* grad_offsets /* host */, float* flat_grad, void* workspace, const float* points,
                    const float* aux, void* stream);
int hn_mlp_bwd_weights(const hn_model_desc* desc, const void* saved, int64_t B, int S, int level,
                       const int64_t* grad_offsets /* host */, float* flat_grad, const void* workspace, void* stream);

/* Trunk-only evaluation of one level: the template NeRF — positional encoding of the warped point and the hyper
 * coordinates, trunk, bottleneck, rgb / alpha heads (NerfMLP modules.py:172-298, query_template models.py:447-493) — for
 * rows whose (3 + H) warped point / hyper coordinates are given.  NerfModel.forward (models.py:745-767) re-evaluates the
 * shared TranslationField / HyperSheetMLP at the coarse depths the fine level inherits (`sort(cat[z_coarse, z_new])`); the
 * drop-in model takes those rows' warp-field outputs from the coarse pass instead and runs them through this entry point.
 * It is also the whole network of a model without warp (warped_in = the raw sample points, models.py:568-569).  Same stash
 * / workspace sizes as hn_mlp_fwd / hn_mlp_bwd (the warp / sheet slabs stay unused).
 *   hn_mlp_fwd_trunk  warped_in (B,S,3+H), in launch order -> sigma, rgb (and, if `warped` != NULL, a copy of warped_in)
 *                     at the rows' positions (pos / S_full as in hn_mlp_fwd)
 *   hn_mlp_bwd_trunk  data + weight gradients of the trunk / heads into flat_grad, and g_warped_in (B,S,3+H) =
 *                     d loss / d warped_in (+ g_warped at the rows' positions when given), to be added to the upstream
 *                     gradient of whoever produced warped_in.  ids: NULL unless the template is GLO-conditioned. */
int hn_mlp_fwd_trunk(const hn_model_desc* desc, const void* packed, const float* warped_in, const float* viewdirs,
                     const int64_t* ids, const float* noise, float noise_std, int64_t B, int S, const int32_t* pos,
                     int S_full, float* sigma, float* rgb, float* warped, void* saved, void* stream);
int hn_mlp_bwd_trunk(const hn_model_desc* desc, const void* packed, const int64_t* ids, const float* sigma, const float* rgb,
                     const float* warped_in, const void* saved, const float* g_sigma, const float* g_rgb,
                     const float* g_warped, int64_t B, int S, const int32_t* pos, int S_full, int level,
                     const int64_t* grad_offsets /* host */, float* flat_grad, float* g_warped_in, void* workspace,
                     void* stream);
/* hn_mlp_bwd_trunk split like hn_mlp_bwd_data / hn_mlp_bwd_weights (same workspace hand-off). */
int hn_mlp_bwd_trunk_data(const hn_model_desc* desc, const void* packed, const int64_t* ids, const float* sigma,
                          const float* rgb, const float* warped_in, const void* saved, const float* g_sigma, const float* g_rgb,
                          const float* g_warped, int64_t B, int S, const int32_t* pos, int S_full, int level,
                          const int64_t* grad_offsets /* host */, float* flat_grad, float* g_warped_in, void* workspace,
                          void* stream);
int hn_mlp_bwd_trunk_weights(const hn_model_desc* desc, const void* saved, int64_t B, int S, int level,
                             const int64_t* grad_offsets /* host */, float* flat_grad, const void* workspace, void* stream);

/* Annealed positional encodings (the Nerfies / HyperNeRF coarse-to-fine window).  Band k of an encoder with bands
 * 0..F-1 is scaled by w_k(alpha) = 0.5 (1 - cos(pi clamp(alpha - k, 0, 1))); identity, GLO, view-direction columns, biases
 * and padding never are.  A window on an encoded input is a per-column scale of the weights that read it,
 * W (w . pe) = (W diag(w)) pe, so:
 *   hn_pack_weights_windowed           packs W diag(w) into the forward AND the transposed (data-gradient) images;
 *   hn_mlp_bwd_weights_windowed /      the weight gradient of such a blob: the stash holds the unwindowed encoding, so the
 *   hn_mlp_bwd_trunk_weights_windowed  accumulated dY^T pe is scaled by w on its way to flat_grad (bias sums unchanged).
 * A windowed blob must be paired with the windowed weight-gradient entries, with the same pe_alpha values.
 * pe_alpha: DEVICE array of 4 floats {warp_alpha, hyper_sheet_alpha, nerf_alpha, hyper_alpha}, read by the kernels (a CUDA
 * graph replays with new values without a new capture); +inf (or any alpha >= F) = no window.  Encoders:
 *   warp_alpha         posenc_orig(points, 10) of the TranslationField (bands of 6 columns after the 3 identity columns),
 *                      posenc(points, 0, 8) of the SE3Field (48 columns, bands of 6)
 *   hyper_sheet_alpha  posenc_orig(points, 7) of the HyperSheetMLP
 *   nerf_alpha         posenc_orig(warped xyz, xyz_freqs) of both levels' trunks
 *   hyper_alpha        posenc_orig(hyper point, hyper_freqs) of both levels' trunks (bands of 2H columns after H identity)
 * An alpha whose encoder the configuration does not have is not read.  The static NeRF has no window (-13). */
int hn_pack_weights_windowed(const hn_model_desc* desc, const float* flat_params, const int64_t* param_offsets /* host */,
                             int level, void* packed, const float* pe_alpha, void* stream);
int hn_mlp_bwd_weights_windowed(const hn_model_desc* desc, const void* saved, int64_t B, int S, int level,
                                const int64_t* grad_offsets /* host */, float* flat_grad, const void* workspace,
                                const float* pe_alpha, void* stream);
int hn_mlp_bwd_trunk_weights_windowed(const hn_model_desc* desc, const void* saved, int64_t B, int S, int level,
                                      const int64_t* grad_offsets /* host */, float* flat_grad, const void* workspace,
                                      const float* pe_alpha, void* stream);

/* Warp-stage-only evaluation (level-0 blob as hn_pack_weights[_windowed] packed it): the TranslationField + HyperSheetMLP
 * (warping.py:28-125, modules.py:302-337; or the axis-aligned hyper point, models.py:533-534) or the SE3Field
 * (warping.py:128-272) that hn_mlp_fwd runs ahead of the template, without the template behind it.  `warped` is
 * bit-identical to hn_mlp_fwd's `warped` output for the same points, ids, blob and mode (inference / training).
 *   hn_mlp_fwd_warp          points (B,S,3), ids (B,) -> warped (B,S,3+H); saved (hn_sizes.warp_saved_bytes; NULL =
 *                            inference); aux: SE3 only, (B,S,6) screw parameters (w, v), required with a stash
 *   hn_mlp_bwd_warp_data     g_warped (B,S,3+H) -> pre-activation gradients in `workspace` (hn_sizes.warp_workspace_bytes)
 *                            and the GLO-table gradient; points / aux: SE3 only, as the forward saw / wrote them.  The
 *                            sample points take no gradient.
 *   hn_mlp_bwd_warp_weights  dW / db of the warp / sheet tensors into flat_grad; pe_alpha: NULL for an unwindowed blob, else
 *                            the device alphas the blob was packed with (hn_pack_weights_windowed).
 * A static descriptor or one without warp is rejected (-13); B and S must be positive. */
int hn_mlp_fwd_warp(const hn_model_desc* desc, const void* packed, const float* points, const int64_t* ids, int64_t B, int S,
                    float* warped, void* saved, float* aux, void* stream);
int hn_mlp_bwd_warp_data(const hn_model_desc* desc, const void* packed, const int64_t* ids, const void* saved,
                         const float* g_warped, int64_t B, int S, const int64_t* grad_offsets /* host */, float* flat_grad,
                         void* workspace, const float* points, const float* aux, void* stream);
int hn_mlp_bwd_warp_weights(const hn_model_desc* desc, const void* saved, int64_t B, int S,
                            const int64_t* grad_offsets /* host */, float* flat_grad, const void* workspace,
                            const float* pe_alpha, void* stream);

/* compute_background_loss + utils.general_loss_with_squared_residual of the JAX HyperNeRF (hypernerf/training.py): the
 * torch port has no counterpart (its losses.py has the MSE only), so the formula is restated (DESIGN.md §2c).  For n
 * points with warped outputs (n, warped_cols) and the jittered inputs points (n, 3):
 *   r^2 = sum_{c<3} (warped_c - points_c)^2,  rho = (b / a) ((r^2 / scale^2 / b + 1)^(a/2) - 1),
 *   b = max(eps, |alpha - 2|), a = sign(alpha) max(eps, |alpha|) (sign(0) = +1), eps = FLT_EPSILON;
 *   sums[0] += sum rho (caller zeroes it);  g_warped[:, :3] = grad_scale d rho / d r^2 2 (warped - points),
 *   g_warped[:, 3:] = 0 (g_warped may be NULL).  n must be positive, scale positive. */
int hn_background_loss(const float* warped, const float* points, int64_t n, int warped_cols, float alpha, float scale,
                       float grad_scale, float* sums, float* g_warped, void* stream);

/* Jacobian of the translation warp, jac[b, s, r, c] = d warped_r / d points_c (r, c < 3), for the nerfies elastic loss
 * (DESIGN.md §2e).  The forward is the bias-free gated linear pass of the warp stage along each input direction c,
 * masked by the ReLU gates of the primal's warp-only stash `primal_saved` (hn_mlp_fwd_warp with the same blob, points,
 * ids, B, S and a stash).  tangent_saved (3 x hn_sizes.warp_saved_bytes, plane c at c x warp_saved_bytes; NULL = Jacobian
 * only) receives each plane's X slabs in the warp-only stash layout, gate words unwritten.  The backward of a dL/dJ = G
 * is, per plane c: hn_mlp_bwd_warp_data on `primal_saved` with g_warped = (G[:, :, c], 0_H) (its GLO-table output is
 * not a gradient: point it at a scratch table), then hn_mlp_bwd_warp_weights on plane c of tangent_saved with the GLO
 * and every bias offset set to -1 (biases, the GLO table and the sheet take no gradient from J).
 * SE3, static and no-warp descriptors are rejected (-13); B and S must be positive. */
int hn_mlp_fwd_warp_tangent(const hn_model_desc* desc, const void* packed, const float* points, const void* primal_saved,
                            int64_t B, int S, float* jac, void* tangent_saved, void* stream);

/* compute_elastic_loss of Nerfies (loss_type 'log_svals') + general_loss_with_squared_residual, for n samples with
 * Jacobians jac (n, 3, 3) and rendering weights (n):
 *   r^2 = sum_i log^2 max(sigma_i(J), eps),  rho(r^2) as in hn_background_loss;  sums[0] += sum w rho (caller zeroes it);
 *   g_planes (3, n, 3 + hyper_cols): plane c, columns r < 3 = grad_scale w d rho / d r^2 (d r^2 / dJ)[r, c], the hyper
 *   columns 0 (NULL: no gradient) — the g_warped planes of the tangent backward.
 * n must be positive, scale and eps positive, hyper_cols >= 0. */
int hn_elastic_loss(const float* jac, const float* weights, int64_t n, float alpha, float scale, float eps, float grad_scale,
                    float* sums, float* g_planes, int hyper_cols, void* stream);

/* losses.py:9-14 (MSELoss: mean-MSE of coarse.rgb + fine.rgb against the target colours) fused with its gradient seed and
 * with the fine-level MSE of metrics.py:4-13 (psnr = -10 log10(mse)).  sums[0] += sum (coarse - t)^2, sums[1] += sum
 * (fine - t)^2 (caller zeroes `sums`); g_level (B,3) = 2 (pred - t) * grad_scale, grad_scale = upstream / (3 B_global).
 * rgb_fine / g_coarse / g_fine may be NULL. */
int hn_mse_loss(const float* rgb_coarse, const float* rgb_fine, const float* targets, int64_t B, float grad_scale, float* sums,
                float* g_coarse, float* g_fine, void* stream);

/* datasets/ray_utils.py:5-93 (get_ray_directions, get_rays, get_ndc_rays) + the ray-row layout of datasets/llff.py:316-332 for
 * one H x W frame on the device: rays (H*W, cols) = [origin(3), direction(3), near = 0, far = 1 (, image id)], cols = 8
 * or 9.  c2w_host: HOST pointer to the (3,4) row-major camera-to-world matrix. */
int hn_make_ndc_rays(int H, int W, float focal, const float* c2w_host, float near_plane, float image_id, int cols,
                     float* rays, void* stream);

/* utils/__init__.py:22-41 (get_optimizer: torch.optim.Adam(parameters, lr, eps=1e-8, weight_decay)) — one Adam.step over the
 * flat fp32 buffers (parameters, gradient, exp_avg, exp_avg_sq; n floats each, 16-byte aligned) in a single launch:
 *   g = grads * grad_scale + weight_decay * p;  m += (g - m)(1 - beta1);  v = beta2 v + (1 - beta2) g^2;
 *   p -= lr / (1 - beta1^step) * m / (sqrt(v) / sqrt(1 - beta2^step) + eps)            (step counts from 1)
 * grad_scale folds the 1/world_size of a summed all-reduce (or an AMP loss scale) into the same pass. */
int hn_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1,
                 float beta2, float eps, float weight_decay, int64_t step, float grad_scale, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HYPERNERF_B200_H */
