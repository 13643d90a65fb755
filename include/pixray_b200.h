/* pixray_b200 -- C ABI of the B200-native engine for pixray's per-iteration hot path.
 *
 * Plain C: pointers and sizes only, no torch types.  Every entry point below replaces one method the reference's
 * Python loop calls each iteration (file:line are relative to the reference checkout, pixray/pixray @ 37b03cf):
 *
 *   pxr_synth          <- drawer.synth(cur_iteration)          pixray.py:1206, vqgan.py:190-195, fast_pixeldrawer.py:89-91,
 *                                                              fftdrawer.py:78-84, vdiff.py:159-172
 *   pxr_make_cutouts   <- MakeCutouts.forward(out)             pixray.py:445-511 (cached-transform semantics 480-486)
 *   pxr_encode_image   <- CLIP_Base.encode_image(cutouts)      slip.py:21-42, 52-66
 *   pxr_prompt_loss    <- Prompt.forward(embeds) per prompt    pixray.py:268-280 (spherical_dist_loss 262-265)
 *   pxr_backward       <- sum(lossAll).backward()              pixray.py:1481-1482
 *   pxr_step           <- opt.step(); drawer.clip_z()          pixray.py:1484-1487, 538-539, vqgan.py:202-204
 *   pxr_iterate        <- one pass of train()                  pixray.py:1436-1512 (ascend_txt 1243-1406)
 *
 * Conventions: functions return 0 on success and a negative code on failure; pxr_last_error() gives the message.
 * All work is enqueued on ONE engine-owned CUDA stream; only pxr_sync, pxr_read_* and the *_host variants block.
 * A handle is owned by one host thread (the reference keeps its session in module globals, pixray.py:1022-1063:
 * one session per process, not re-entrant).  Buffers passed in are device pointers unless the name says host;
 * layouts at the boundary are the reference's: NCHW fp32 images, [cutn, D] fp32 embeddings.
 * There is no CPU fallback: without a CUDA device pxr_create fails.
 */
#ifndef PIXRAY_B200_H
#define PIXRAY_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct pxr_engine* pxr_handle;

enum { PXR_DRAWER_VQGAN = 0, PXR_DRAWER_PIXEL = 1, PXR_DRAWER_FFT = 2, PXR_DRAWER_VDIFF = 3 };
enum { PXR_PAD_REFLECTION = 0, PXR_PAD_BORDER = 1, PXR_PAD_ZEROS = 2 };
enum { PXR_DTYPE_F16 = 0, PXR_DTYPE_BF16 = 1 };
/* optimiser kinds for pxr_set_optimizer (args.optimiser, pixray.py:536-553; library defaults, only lr is set) */
enum { PXR_OPT_ADAM = 0, PXR_OPT_ADAMW = 1, PXR_OPT_ADAGRAD = 2, PXR_OPT_ADAMAX = 3, PXR_OPT_DIFFGRAD = 4 };
/* module ids for pxr_load_weight */
enum { PXR_MOD_VQGAN = 0, PXR_MOD_CLIP0 = 1, PXR_MOD_CLIP1 = 2 };

typedef struct {
  int width;     /* transformer width (768 for ViT-B) */
  int layers;    /* 12 */
  int heads;     /* 12 */
  int patch;     /* 16 or 32 */
  int image_res; /* 224 == MakeCutouts cut_size (pixray.py:643-649) */
  int out_dim;   /* 512 */
} pxr_clip_cfg;

typedef struct {
  int device;            /* CUDA ordinal */
  int rank, world;       /* cutout-shard rank / number of ranks (1 = single GPU) */
  int drawer;            /* PXR_DRAWER_* */
  int image_h, image_w;  /* canvas (vqgan: multiple of 16) */
  /* taming Decoder hyper-parameters (vqgan.py:122-142: model.decoder / model.quantize) */
  int z_channels, n_embed, ch, num_res_blocks, attn_resolution, n_levels, resolution;
  int ch_mult[8];
  /* pixel drawer grid (fast_pixeldrawer.py:37-63) */
  int grid_rows, grid_cols;
  /* MakeCutouts(cut_size, cutn) pixray.py:400-443; cutn is the GLOBAL count, this rank owns a slice */
  int cutn, cut_size;
  int n_clip;
  pxr_clip_cfg clip[2];
  float noise_fac;       /* pixray.py:439 (0.1) */
  uint64_t seed;
  int op_dtype;          /* PXR_DTYPE_*: tensor-core operand type (accumulation is always fp32) */
  float grad_scale;      /* backward runs on grad_scale * dL (fp16 range management); 0 = default */
  float beta1, beta2, adam_eps; /* optim.Adam defaults 0.9 / 0.999 / 1e-8 when 0 */
  /* fft drawer (fftdrawer.py:16-22, 57-61): fft_image(decay_power) / to_valid_rgb(colors) / image_f(contrast) */
  float fft_decay, fft_colors, fft_contrast; /* 0 -> 1.5 / 1.5 / 0.9 */
  /* global_aspect_width = args.size[0] / args.size[1] (pixray.py:1931): != 1 stretches the pooled cut_size x cut_size image
   * to [cut_size, int(cut_size * a)] (a > 1) or [int(cut_size / a), cut_size] (a < 1) before the warps (pixray.py:468-472)
   * and changes the wide stack's affine (pixray.py:420-432).  0 = 1 (square). */
  float cut_aspect;
  /* the stretched size itself, int(cut_size * a) resp. int(cut_size * (1 / a)) as the reference's Python floats give it
   * (kornia rescale truncates); 0 = derive from cut_aspect (which, being a C float, can round across an integer) */
  int cut_src_h, cut_src_w;
  int reserved[2];
} pxr_config;

/* Per-iteration cutout parameters (SURVEY.md Appendix A): what kornia's augmentations sample per cutout, made explicit.
 * transforms[cutn*9]: row-major 3x3 "dst_pix <- src_pix" homographies exactly as MakeCutouts.transforms caches them
 * (pixray.py:498; src = the pooled image, stretched when cut_aspect != 1); indices [0, int(0.6*cutn)) form the zoom group, the rest the wide group (pixray.py:407, 493-494). */
typedef struct {
  const float* transforms; /* host, [cutn, 3, 3] */
  int zoom_padding;        /* PXR_PAD_REFLECTION on even iterations, PXR_PAD_BORDER on odd (pixray.py:1250-1253) */
  float fill;              /* wide-group fill grey = random.random() (pixray.py:1255-1258) */
  /* batch + facs * randn_like(batch) (pixray.py:508-510).  Given together: replayed as is.  Both NULL: with
   * transforms == NULL the engine draws them (Philox keyed by seed, iteration and GLOBAL element index), with explicit
   * transforms the call is a deterministic replay WITHOUT noise.  One without the other is an error (-61). */
  const float* noise_facs; /* host, [cutn] ~ U(0, noise_fac) (pixray.py:509) */
  const float* noise;      /* DEVICE, [cutn,3,cs,cs] standard normal (pixray.py:510) */
  /* K.ColorJitter(hue=0.1, saturation=0.1, p=0.8), the last stage of both stacks (pixray.py:416, 436): host
   * [cutn, 3] rows {code, saturation_factor, hue_factor}.  code 0 = this cutout missed the Bernoulli(p); else
   * 256 + o0 + 4*o1 + 16*o2 + 64*o3 with o_k the transform applied k-th (0 brightness, 1 contrast, 2 saturation,
   * 3 hue: kornia's params["order"]).  NULL with explicit transforms = no jitter (the cached-transform replay,
   * pixray.py:480-486); with transforms == NULL the engine draws these too (pxr_set_color_jitter). */
  const float* color_jitter;
} pxr_cut_params;

const char* pxr_last_error(pxr_handle h); /* h may be NULL for creation errors */
const char* pxr_version(void);

int pxr_create(const pxr_config* cfg, pxr_handle* out);
void pxr_destroy(pxr_handle h);

/* Weights by the reference's state_dict key (e.g. "decoder.conv_in.weight", "quantize.embedding.weight",
 * "visual.transformer.resblocks.0.attn.in_proj_weight").  data: fp32, host or device; copied and repacked. */
int pxr_load_weight(pxr_handle h, int module_id, const char* name, const float* data, const int64_t* dims, int ndim);
/* After all weights: builds every kernel plan / workspace.  Fails listing the first missing weight. */
int pxr_finalize(pxr_handle h);

/* Prompt(embed, weight, stop) list of one perceptor (pixray.py:859-915).  embeds host [n, D]. */
int pxr_set_prompts(pxr_handle h, int clip_idx, const float* embeds, int n, int D, const float* weights,
                    const float* stops);

/* Image prompts (pixray.py:1308-1336, pmsImageTable): imgs host or device fp32 [n, 3, H, W] in [0, 1] at the output
 * size (copied).  Every iteration -- inside pxr_iterate / pxr_make_cutouts, before the main pass -- each image is cut
 * with that iteration's cached transforms (no ColorJitter on the cached path, pixray.py:480-486; fresh noise, or the
 * explicit noise of pxr_cut_params replayed), encoded by every perceptor, and scored as a throwaway
 * Prompt(embed [cutn, D], weights[k]) (weights NULL = 1, args.image_prompt_weight otherwise) whose loss follows that
 * perceptor's text prompts in the loss vector.  Cutout-sharded ranks exchange the [cutn, D] rows (one allreduce).
 * n = 0 clears. */
int pxr_set_image_prompts(pxr_handle h, const float* imgs, int n, const float* weights);
/* the same with every target at its own size: imgs[k] fp32 [3, hs[k], ws[k]] (resize_image keeps the source aspect and never
 * upsamples, pixray.py:514-518; MakeCutouts pools any size to cut_size x cut_size, pixray.py:463) */
int pxr_set_image_prompts_sized(pxr_handle h, const float* const* imgs, const int* hs, const int* ws, int n,
                                const float* weights);

/* Spot prompts (args.spot_prompts / spot_prompts_off: pixray.py:917-931, 1262-1293; mask from fetch_spot_indexes 370-394,
 * applied to the pooled image at 453-459).  which = 1: `embeds` are scored on cutouts of the image with the SPOT zeroed
 * (make_cutouts(out, spot=1) zeroes mask >= 0.5), which = 0: with everything but the spot zeroed.  Every pxr_iterate then
 * runs one more cutout + encode + backward pass per kind (cached transforms of the iteration, no ColorJitter, fresh noise);
 * their losses come FIRST in the perceptor's part of the loss vector (spot, spot off, prompts, image prompts).
 * mask: host bytes [3, cut_size, cut_size], != 0 where the resized RGB mask image is >= 0.5. */
int pxr_set_spot_prompts(pxr_handle h, int clip_idx, int which, const float* embeds, int n, int D, const float* weights,
                         const float* stops);
int pxr_set_spot_mask(pxr_handle h, const unsigned char* mask);

/* Multi-GPU: 128-byte ncclUniqueId from rank 0; the engine owns the communicator. */
int pxr_set_comm(pxr_handle h, const void* nccl_unique_id, int rank, int world);
int pxr_get_unique_id(void* out128);

int pxr_synth(pxr_handle h, const float* z, float* out_img /* [3,H,W] */);
/* z = model.encode(img)[0]: VqganDrawer.init_from_tensor / reapply_from_tensor / get_z_from_tensor (vqgan.py:174-185) --
 * taming Encoder + quant_conv + nearest codebook row.  img device [3,H,W] in [-1,1]; z_out device [z_channels,h,w].
 * Available when the weights loaded before pxr_finalize include the checkpoint's encoder.* and quant_conv.* tensors. */
int pxr_vqgan_encode(pxr_handle h, const float* img, float* z_out);
/* Distribution of the engine-drawn ColorJitter: Bernoulli(p) per cutout, saturation_factor ~ U(1-s, 1+s),
 * hue_factor ~ U(-hue, hue), one random order per group and iteration.  Defaults = the reference's call sites
 * (0.8, 0.1, 0.1); p = 0 turns the stage off. */
int pxr_set_color_jitter(pxr_handle h, float p, float saturation, float hue);
int pxr_make_cutouts(pxr_handle h, const float* img, const pxr_cut_params* p, int iter,
                     float* out_batch /* [cutn_local,3,cs,cs] */);
int pxr_encode_image(pxr_handle h, int clip_idx, const float* batch, float* out_embeds /* [cutn_local, D] */);
int pxr_prompt_loss(pxr_handle h, int clip_idx, const float* embeds, float* out_losses /* [n_prompts] */);
int pxr_backward(pxr_handle h, float* z_grad);
int pxr_step(pxr_handle h, float* z, float lr, int iter);
int pxr_iterate(pxr_handle h, float* z, float lr, int iter, const pxr_cut_params* p,
                float* out_losses_host /* pinned or pageable; may be NULL */);
/* Auxiliary losses: Losses/*.py behind LossInterface.get_loss, summed into the iteration's loss list by ascend_txt
 * (pixray.py:1384-1393, custom_loss spec "name:weight").  Each becomes one more entry of the loss vector (after the
 * prompts, in the order added) and one more term of the gradient.  params (host floats), by kind:
 *   SYMMETRY   {symmetry_weight}                                            Losses/SymmetryLoss.py:14-17   (image)
 *   SATURATION {saturation_weight}                                          Losses/SaturationLoss.py:15-30 (cutouts)
 *   PALETTE    {palette_weight, r0,g0,b0, r1,g1,b1, ...}  colours in [0,1]  Losses/PaletteLoss.py:25-35    (cutouts)
 *   SMOOTHNESS {smoothness_weight, type (0 default, 1 clipped, 2 log), spacing}   Losses/SmoothnessLoss.py:89-108
 *   EDGE       {edge_color_weight, global_color_weight, left,right,upper,lower (pixels), r,g,b}  Losses/EdgeLoss.py:60-108
 *   GAUSSIAN   {gaussian_weight, std_y, std_x, R,G,B (0..255)}              Losses/GaussianLoss.py:31-44   (image)
 *   AESTHETIC  {aesthetic_target, bias, w[D]}  linear head on the last perceptor's embeddings  Losses/AestheticLoss.py:30-33 */
enum { PXR_LOSS_SYMMETRY = 0, PXR_LOSS_SATURATION = 1, PXR_LOSS_PALETTE = 2, PXR_LOSS_SMOOTHNESS = 3, PXR_LOSS_EDGE = 4,
       PXR_LOSS_GAUSSIAN = 5, PXR_LOSS_AESTHETIC = 6 };
int pxr_add_aux_loss(pxr_handle h, int kind, float weight, const float* params, int n_params);
int pxr_clear_aux_losses(pxr_handle h);

/* Anchors to a stored copy: the init_weight family and image_labels of ascend_txt (pixray.py:1344-1375).  Each is one entry
 * of the loss vector after the prompts and before the auxiliary losses, in the order added (the reference's order is
 * image_labels..., init_weight, init_weight_dist, init_weight_pix, init_weight_cos).
 *   SPHERICAL  spherical_dist_loss(z.reshape(1,-1), ref.reshape(1,-1)) * weight      init_weight, image_label_weight
 *   MSE        F.mse_loss(z, ref) * weight / 2                                        init_weight_dist
 *   COS        F.cosine_embedding_loss(z.reshape(1,-1), ref.reshape(1,-1), 1) * weight  init_weight_cos
 *   PIX        F.l1_loss(out, ref) * weight / 2, ref = init_image_tensor [3,H,W] in [0,1]   init_weight_pix
 * `ref` (host or device floats) is copied: the latent's element count for the first three (z_orig = drawer.get_z_copy(),
 * pixray.py:719, or an encoded label image), 3*H*W of the image MakeCutouts sees for PIX.  The latent terms add to z.grad
 * after the drawer backward; PIX adds to the image gradient before it.  Replicated on every rank when sharded. */
enum { PXR_ANCHOR_SPHERICAL = 0, PXR_ANCHOR_MSE = 1, PXR_ANCHOR_COS = 2, PXR_ANCHOR_PIX = 3 };
int pxr_add_anchor(pxr_handle h, int kind, float weight, const float* ref, long long n);
int pxr_clear_anchors(pxr_handle h);
int pxr_num_losses(pxr_handle h, int* out); /* filters + prompts of every perceptor + auxiliary losses */

/* Filters (args.filters "name:weight,..."; FilterInterface.forward(img) -> (img, loss), pixray.py:651-668, applied to the
 * drawer's output before MakeCutouts in do_synth_and_filter, pixray.py:1203-1222).  Inside pxr_iterate only.  params:
 *   TILER     {}                                               filters/tiler.py: torch.roll by random (h, w) shifts
 *   WALLPAPER {type (0 none, 1 shift, 2 horizontal, 3 vertical), wallpaper_edge_match}   filters/wallpaper.py
 *   LOOKUP    {lookup_beta, r0,g0,b0, ...} palette in [0,1]     filters/colorlookup.py (nearest colour, straight-through)
 * Each filter owns one entry at the FRONT of the loss vector (its weighted loss; 0 for the loss-free ones).  The random
 * shifts are engine-drawn per iteration (Philox by seed / iteration) or fixed through pxr_set_filter_shifts. */
enum { PXR_FILTER_TILER = 0, PXR_FILTER_WALLPAPER = 1, PXR_FILTER_LOOKUP = 2 };
int pxr_add_filter(pxr_handle h, int kind, float weight, const float* params, int n_params);
int pxr_clear_filters(pxr_handle h);
int pxr_set_filter_shifts(pxr_handle h, int filter_idx, int rand_h, int rand_w);
int pxr_read_losses(pxr_handle h, float* out_host); /* blocking: the loss vector of the last forward / backward */

/* vdiff drawer (PXR_DRAWER_VDIFF; VdiffDrawer, vdiff.py:58-190, over diffusion/models/cc12m_1.py).  z = x [1,3,H,W];
 * weights under the checkpoint's own keys through pxr_load_weight(module PXR_MOD_VQGAN = the drawer slot).
 *   set_schedule : sample_state's steps / alphas / sigmas (vdiff.py:113-126, sampling.py:41-51), n = iterations + 1
 *   set_clip_embed: extra_args["clip_embed"] (pixray.py:880-885), host [512]
 *   set_iteration: the schedule index the per-op pxr_synth uses (pxr_iterate uses its own `iter`)
 *   renoise      : drawer.makenoise(cur_it) (vdiff.py:156-157, sampling.sample_step_noise 18-39) on the pred / v the last
 *                  synth kept; noise: device [3,H,W] standard normal (torch.randn_like), or NULL for eta = 0 */
int pxr_vdiff_set_schedule(pxr_handle h, const float* steps, const float* alphas, const float* sigmas, int n);
int pxr_vdiff_set_clip_embed(pxr_handle h, const float* embed, int D);
int pxr_vdiff_set_iteration(pxr_handle h, int i);
int pxr_vdiff_renoise(pxr_handle h, float* z, int i, const float* noise);

int pxr_reset_optimizer(pxr_handle h); /* rebuild_optimisers: fresh state of the current optimiser (pixray.py:520-555, 1511) */
/* rebuild_optimisers with another args.optimiser: selects PXR_OPT_* `kind` (Adam after pxr_create), then does exactly
 * what pxr_reset_optimizer does.  Every later pxr_step / pxr_iterate steps that optimiser. */
int pxr_set_optimizer(pxr_handle h, int kind);

/* train()'s control decisions on the device (checkdrop pixray.py:1090-1109; scheduled learning-rate drops, auto-stop and
 * rebuild_optimisers 1464-1512): the optimiser step of every pxr_iterate reads the iteration's loss vector, tracks the best
 * loss, drops the learning rate (fresh Adam at base_lr / 10^drops) at the iterations in `drops` or -- with auto_stop --
 * when the loss has not improved for iter_drop_delay iterations, and stops updating z once max_loss_drops is exceeded.
 * No host synchronisation: pxr_iterate's `lr` is ignored afterwards and pxr_poll_status reads the last completed
 * iteration's record from pinned memory. */
typedef struct {
  int iter;            /* the iteration this record describes */
  float loss_sum;      /* sum(lossAll) of that iteration */
  float best_loss;     /* after the iteration (1e20 right after a rebuild) */
  int best_iter, num_loss_drop;
  int stopped;         /* train() would have returned False: later iterations leave z untouched */
  int rebuilt;         /* the iteration ended with rebuild_optimisers */
  float lr;            /* learning rate the NEXT iteration uses */
  int n_losses;
  float losses[64];
} pxr_status;
int pxr_set_schedule(pxr_handle h, float base_lr, int iter_drop_delay, int max_loss_drops, int auto_stop, const int* drops,
                     int n_drops);
int pxr_poll_status(pxr_handle h, pxr_status* out); /* 0 ok, 1 no consistent record yet; never blocks */
/* args.batches (pixray.py:1464-1482): every pxr_iterate runs this many ascend_txt + backward passes with fresh
 * engine-drawn augmentations, accumulates z.grad over them and takes ONE optimiser step */
int pxr_set_batches(pxr_handle h, int batches);
/* hand pxr_step the gradient to apply (device [z_numel]); the per-op plugin loop accumulates several passes itself */
int pxr_set_z_grad(pxr_handle h, const float* z_grad);
int pxr_sync(pxr_handle h);

/* Checkpoint of the optimisation state for resume (SURVEY.md 8f-3): {z, optimiser state m, v (+ DiffGrad's previous
 * gradient), optimiser kind, step count, learning-rate / best-loss / drop bookkeeping} as one host blob of pxr_state_size
 * bytes (the size depends on the current optimiser kind).  Load into an engine of the same configuration and optimiser
 * kind (after pxr_set_schedule when the saved session was device-managed) and keep calling pxr_iterate with the next
 * iteration number: the engine-drawn augmentations are keyed by (seed, iteration), so the continuation follows the
 * uninterrupted run. */
int pxr_state_size(pxr_handle h, int64_t* nbytes);
int pxr_save_state(pxr_handle h, void* host_buf);
int pxr_load_state(pxr_handle h, const void* host_buf);

/* Introspection used by tests and bench.py */
int pxr_num_kernel_launches(pxr_handle h, int64_t* out); /* launches issued since create */
/* one iteration with CUDA events around every launch: out6 = {gemm ms, gemm launches, gemm algorithmic FLOPs,
 * other ms, other launches, whole-iteration ms}; feeds bench.py's roofline object */
int pxr_profile_iteration(pxr_handle h, float* z, float lr, int iter, double* out6);
/* the same, plus the compulsory (algorithmic) bytes of the tensor-core launches: each operand read once, each epilogue
 * tensor read / written once -- the denominator against which measured DRAM traffic shows wasted re-reads */
int pxr_profile_iteration2(pxr_handle h, float* z, float lr, int iter, double* out6, double* tensor_bytes);
int pxr_get_stream(pxr_handle h, void** out);
int pxr_z_numel(pxr_handle h, int64_t* out);
int pxr_z_bounds(pxr_handle h, float* zmin, float* zmax); /* device [z_channels]: codebook per-channel min/max */

/* ---------------------------------------------------------------- test hooks (used only by tests/) */
/* copy a named internal buffer (e.g. "g_img", "batch", "clip0.gx") to `out` (host or device) */
int pxr_debug_read(pxr_handle h, const char* name, void* out, int64_t nbytes);

typedef struct {
  const void* a;
  int a_mode; /* 0 K-major, 1 MN-major */
  long long lda, a_mn_extent, a_k_extent, a_bs0, a_bs1;
  const void* b;
  int b_mode, b_batched;
  long long ldb, b_mn_extent, b_k_extent, b_bs0, b_bs1;
  int nb0, nb1;
  int M, N, K, block_n, fmt;
  float alpha;
  const float* bias;
  int bias_per_row, act;
  const void* aux_in;
  void* aux_out;
  const float* res_f32;
  const void* res_f16;
  float* out_f32;
  void* out_f16;
  long long ldc, c_bs0, c_bs1;
  void* stream;
  int repeat;
  int n_store; /* fused-softmax epilogues (act 3 / 4): zero-fill columns [N, n_store) */
  int cta_group; /* 0 auto, 1 single-CTA tiles, 2 CTA pairs (tcgen05 cta_group::2) */
  int tma_epi;   /* 0 auto (tensor-map epilogue when the tensors allow it), -1 force the generic epilogue */
} pxr_test_gemm_desc;

int pxr_test_gemm(const pxr_test_gemm_desc* d, char* err, int errlen);
/* implicit-GEMM conv over NHWC fp16: d->a = input (pixel stride lda), d->b = weights [taps*cout_pad, c_in] */
int pxr_test_conv(const pxr_test_gemm_desc* d, int batch, int H, int W, int c_in, int cout_pad, int ksize, char* err,
                  int errlen);

/* host-side evaluation of the ColorJitter pixel body and its vector-Jacobian product (no GPU needed) */
int pxr_test_color_jitter_host(const float* rgb, int n, int code, float saturation, float hue, const float* g_out,
                               float* out, float* g_in);
/* the same body on the device; all pointers are DEVICE [n, 3] (default stream, synchronous) */
int pxr_test_color_jitter_device(const float* rgb, int n, int code, float saturation, float hue, const float* g_out,
                                 float* out, float* g_in);

/* adaptive-pool window bounds as the device computes them (pool_fwd / pool_bwd): DEVICE int [out_size] each */
int pxr_test_pool_bounds(int in_size, int out_size, int* starts, int* ends);

/* fused ViT attention (attn_tc.cu): forward, and backward when d_o != NULL.  qkv [B*T, 3W], o / d_o [B*T, W],
 * gqkv [B*T, 3W] fp16 device tensors, lse [B*H*T] fp32; heads are 64 wide (W = 64 H), T <= 256 */
int pxr_test_attention(const void* qkv, void* o, float* lse, const void* d_o, void* gqkv, int B, int T, int H, int W,
                       float scale, int repeat, char* err, int errlen);

/* GroupNorm(32, C, eps 1e-6)(+ swish) of the VQGAN decoder (taming Normalize + nonlinearity), forward and -- when dy or
 * ws_dy is given -- backward, on DEVICE NHWC fp16 tensors [pixels, C].  variant 0: single-kernel grid-barrier version,
 * 1: one thread-block cluster per group; with ws / ws_dy (variant 1) the kernel is also the epilogue of a split-K
 * convolution (fp32 partial sums [splits][pixels][C]).  scratch: 64 * (num_sms + 2) floats + 8 zeroed bytes. */
int pxr_test_groupnorm(int variant, const void* x, const float* ws, int splits, const float* bias, const void* res,
                       void* x_out, const float* gamma, const float* beta, int pixels, int C, int swish, void* y,
                       float* stats, const void* dy, const float* ws_dy, int splits_dy, const void* dres, void* dx,
                       float* scratch, int repeat);

#ifdef __cplusplus
}
#endif
#endif
