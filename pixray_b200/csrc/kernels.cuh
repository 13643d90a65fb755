// Launchers of the non-GEMM kernels of the hot path (gather / pointwise / reduction; HBM-bound).
// Every launcher enqueues on `st` and returns; none synchronises.  Layouts: decoder activations are NHWC fp16
// ([pixels, C], C a multiple of 64); the CLIP residual stream is fp32 [tokens, W]; images are planar fp32 [3,H,W].
// Gradient tensors in fp16 carry grad_scale * dL (see DESIGN.md "fp16 backward").
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace pxr {

typedef __half act_t;

// ------------------------------------------------------------------ VQGAN drawer (vqgan.py:60-64, 190-195)
// Nearest codebook row per latent position (exact fp32), straight-through output as NHWC fp16.
//   z: [C, hw] fp32 (NCHW of the reference's z with N=1); cbT: [C, n_e] fp32; c2: [n_e] = sum_k cb^2
//   part_d/part_i: scratch [hw, n_chunks]; idx: [hw]; zq: [hw, C] fp16; cb: [n_e, C] fp32
void vq_nearest(const float* z, const float* cbT, const float* c2, const float* cb, int C, int hw, int n_e,
                float* part_d, int* part_i, int* idx, act_t* zq, cudaStream_t st);
// The same search with the hw x n_e dot products on the tensor cores (kernels_vq_tc.cu): vq_prep -> one gemm_tc GEMM
// (zh [hw, C] x cbh [n_e, C]^T -> scores [hw, ld] fp32) -> vq_select, which re-evaluates in exact fp32 every code whose
// approximate distance lies within the rounding bound of the minimum, so the index is the one vq_nearest picks.
// pinfo: [hw][4] = {|x|^2, power-of-two scale, |x|_2, |x|_1}; cb_scale: the power of two the fp16 codebook copy carries;
// cmax2 / cmax1: max_j |c_j|_2, |c_j|_1; stats (may be null): {candidates rechecked, positions that fell back}, cumulative.
bool vq_tc_supported(int C, int n_e);
void vq_prep(const float* z, int C, int hw, act_t* zh, float* pinfo, cudaStream_t st);
void vq_select(const float* scores, int ld, const float* z, const float* cb, const float* c2, const float* pinfo,
               float cb_scale, float cmax2, float cmax1, int C, int hw, int n_e, int* idx, act_t* zq, int* stats,
               cudaStream_t st);
// z_grad[C, hw] fp32 = dzq[hw, C] fp16 / grad_scale   (ReplaceGrad: gradient of z_q goes to z unchanged)
void vq_backward(const act_t* dzq, float inv_scale, int C, int hw, float* z_grad, cudaStream_t st);

// GroupNorm(32, C, eps) [+ swish] over NHWC fp16.  stats: [32][2] (mean, rstd); part: scratch [nblk][32][2].
int gn_num_partials(int pixels, int C);
void gn_stats(const act_t* x, int pixels, int C, float eps, float* part, float* stats, cudaStream_t st);
void gn_apply(const act_t* x, const float* stats, const float* gamma, const float* beta, int pixels, int C, int swish,
              act_t* y, cudaStream_t st);
// dx = GroupNorm'(x) applied to dy (through swish when set) [+ dres]; part2 scratch like gn_stats.
void gn_backward(const act_t* dy, const act_t* x, const float* stats, const float* gamma, const float* beta,
                 int pixels, int C, int swish, const act_t* dres, float* part, float* gstats, act_t* dx,
                 cudaStream_t st);

// The same two operations as ONE kernel each (grid <= one block per SM, grid-wide barrier between the statistics and the apply
// phase, the block's slab of x kept in shared memory): 1 launch and 1 HBM pass instead of 3 launches and 2 passes.
// `part` needs 64 floats per block (<= num_sms blocks).  gn_coop_supported: the slab of a block fits shared memory.
// The grid-wide barrier is a monotonically growing device counter; `issued` mirrors on the host what the launches so far
// will have added, so each launch knows the value it waits for (one GridBarrier per stream).
struct GridBarrier {
  unsigned long long* counter = nullptr;  // device, zero-initialised
  unsigned long long issued = 0;
};
// Variants for the vdiff U-Net (cc12m_1.py:41-50, 78-97): GroupNorm(1, C) (one_group), gamma = modulation scale + 1
// (gamma_add, gamma/beta may be null = 0), activation `swish` argument: 0 none, 1 swish, 2 ReLU, forward residual add.
struct GnOpts {
  int one_group = 0;
  float gamma_add = 0.f;
  const act_t* res = nullptr;  // forward only: y = act(norm(x)) + res
};
bool gn_coop_supported(int pixels, int C, int num_sms);
void gn_forward_coop(const act_t* x, const float* gamma, const float* beta, int pixels, int C, int swish, float eps,
                     float* part, float* stats, act_t* y, int num_sms, GridBarrier* gb, cudaStream_t st,
                     GnOpts o = GnOpts());
void gn_backward_coop(const act_t* dy, const act_t* x, const float* stats, const float* gamma, const float* beta,
                      int pixels, int C, int swish, const act_t* dres, float* part, act_t* dx, int num_sms,
                      GridBarrier* gb, cudaStream_t st, GnOpts o = GnOpts());

// GroupNorm(32, C) with one thread-block cluster per GROUP (kernels_gn_group.cu): no grid-wide barrier, for the layers
// whose group fits the registers of <= 8 CTAs (C/32 in {8, 16, 32} channels per group, pixels * C/256 <= 16384 units).
// `sk` (optional) makes the kernel the epilogue of a split-K convolution as well: forward sums the fp32 partials
// [splits][pixels][ld_ws] (+ bias + res), writes the result to sk->out (pitch C) and normalises it in the same pass;
// backward takes dy from the partials (no bias / res) instead of from memory.
struct GnSplitK {
  const float* ws = nullptr;
  int splits = 0, ld_ws = 0;
  const float* bias = nullptr;
  const act_t* res = nullptr;
  act_t* out = nullptr;
};
bool gn_group_supported(int pixels, int C);  // covered AND inside the size range where it is the faster kernel
bool gn_group_possible(int pixels, int C);   // covered at all (the launchers accept these)
void gn_forward_group(const act_t* x, const GnSplitK* sk, const float* gamma, const float* beta, int pixels, int C,
                      int swish, float eps, float* stats, act_t* y, cudaStream_t st);
void gn_backward_group(const act_t* dy, const GnSplitK* sk, const act_t* x, const float* stats, const float* gamma,
                       const float* beta, int pixels, int C, int swish, const act_t* dres, act_t* dx, cudaStream_t st);

// ---- VQGAN encoder side (taming Encoder; VqganDrawer.init_from_tensor, vqgan.py:174-185): forward only, init time
// image [3, H, W] fp32 in [-1, 1] -> NHWC fp16 [pixels, 64] (channels 3..63 zero: conv_in's padded reduction)
void image_to_nhwc64(const float* img, int pixels, act_t* out, cudaStream_t st);
// taming Downsample: F.pad(x, (0,1,0,1)) + Conv2d(k=3, stride=2, padding=0) == the odd positions of the stride-1 "same"
// convolution: y[i, j] = full[2 i + 1, 2 j + 1], [H, W, C] -> [H/2, W/2, C]
void subsample_odd(const act_t* full, int H, int W, int C, act_t* y, cudaStream_t st);
// z[c, p] = codebook[idx[p], c] (fp32): the quantised latent model.encode returns
void gather_codes(const float* cb, const int* idx, int C, int hw, float* z, cudaStream_t st);

void upsample2x(const act_t* x, int H, int W, int C, act_t* y, cudaStream_t st);        // nearest, [H,W,C]->[2H,2W,C]
void downsum2x(const act_t* gy, int H, int W, int C, act_t* gx, cudaStream_t st);       // adjoint: [2H,2W,C]->[H,W,C]

// conv_out result [pixels, ld] fp32 (3 valid channels) -> image [3, pixels] = clamp((x+1)/2, 0, 1); pre = unclamped.
void image_finish(const float* conv_out, int ld, int pixels, float* pre, float* img, cudaStream_t st);
// ClampWithGrad backward (vqgan.py:76-79) + d/dx of (x+1)/2 -> fp16 [pixels, ld] (ld >= 3; other channels untouched)
void image_finish_backward(const float* g_img, const float* pre, int pixels, int ld, act_t* g_out, cudaStream_t st);

// FastPixelDrawer.synth (fast_pixeldrawer.py:89-91): nearest upsample [3,rows,cols] -> [3,H,W] + clamp; and adjoint.
void pixel_synth(const float* z, int rows, int cols, int H, int W, float* pre, float* img, cudaStream_t st);
void pixel_synth_backward(const float* g_img, const float* pre, int rows, int cols, int H, int W, float inv_scale,
                          float* z_grad, cudaStream_t st);

// ------------------------------------------------------------------ FFT drawer (fftdrawer.py:78-84)
struct FftPlans;  // cuFFT C2R / R2C plans (3 planes of H x W), resolved through dlopen
FftPlans* fft_plans_create(int H, int W, cudaStream_t st, const char** err);
void fft_plans_destroy(FftPlans* p);
// spectrum [3,H,W/2+1,2] -> img [3,H,W] = sigmoid(M (irfft2(scale*spectrum, ortho) * contrast / std)); x, stats kept
void fft_synth_forward(FftPlans* pl, const float* spectrum, const float* scale, const float* M, float contrast,
                       float* scaled, float* x, double* part, float* stats, float* img, cudaStream_t st);
void fft_synth_backward(FftPlans* pl, const float* g_img, const float* img, const float* x, const float* scale,
                        const float* M, float contrast, const float* stats, float* g1, float* G, double* part,
                        float inv_scale, float* z_grad, cudaStream_t st);

// ------------------------------------------------------------------ MakeCutouts (pixray.py:445-511)
// (AdaptiveAvgPool2d + AdaptiveMaxPool2d) / 2 of the whole image, once (pixray.py:463); argmax kept for backward.
void pool_forward(const float* img, int H, int W, int cs, float* pooled, int* argmax, cudaStream_t st);
void pool_backward(const float* g_pooled, const int* argmax, int H, int W, int cs, float* g_img, cudaStream_t st,
                   int accumulate = 0);
// Spot prompts (pixray.py:453-459): cutout[0][mask_indexes] = 0 on the pooled image -- y = keep ? x : 0 with
// keep = (mask[i] != 0) XOR zero_where_set; the same call masks the gradient on the way back (in place when y == x)
void spot_mask_apply(const float* x, const unsigned char* mask, int zero_where_set, int n, float* y, cudaStream_t st);

// kornia.geometry.transform.rescale of the pooled image for non-square canvases (pixray.py:468-472): bilinear,
// align_corners=False ([3, in_h, in_w] -> [3, out_h, out_w]), and its adjoint (g_in must be zeroed by the caller)
void rescale_bilinear(const float* x, int in_h, int in_w, int out_h, int out_w, float* y, cudaStream_t st);
// 64-bit fixed-point accumulation (order-independent sums).  A pass that meets a NaN / Inf / out-of-range contribution
// writes its id to *poison; the conversion to fp32 then yields NaN for the whole tensor (ids only ever grow: no reset).
struct FxPass {
  unsigned int* poison = nullptr;  // device word
  unsigned int pass = 0;           // > 0, unique per accumulate + convert pair on that word
};
// acc: zeroed 64-bit fixed-point accumulator of 3 * in_h * in_w entries (cleared again on return)
void rescale_bilinear_backward(const float* gy, int in_h, int in_w, int out_h, int out_w, long long* acc, FxPass fx, float* gx,
                               cudaStream_t st);

struct CutoutArgs {
  const float* pooled;     // [3, src_h, src_w]: the pooled image (cs x cs), stretched when the canvas is not square
  const float* minv;       // [n_local, 9] src_pix <- dst_pix homographies (device)
  const float* noise_facs; // [n_local]            (noise_mode 1)
  const float* noise;      // [n_local, 3, cs, cs] (noise_mode 1)
  const float* jitter;     // [n_local, 3] {code, saturation_factor, hue_factor} (color_jitter.cuh) or nullptr
  int noise_mode;          // 0 none, 1 explicit facs + noise, 2 engine Philox (seed, iter)
  float noise_fac;         // U(0, noise_fac) upper bound for mode 2 (pixray.py:439)
  int cs, n_local, first_global, cutn_zoom, zoom_padding;
  int src_h, src_w;        // size of `pooled` (== cs, cs on a square canvas)
  float fill;
  uint64_t seed;
  int iter;
};
int cutout_num_blocks(int n_local, int cs);
// batch [n_local,3,cs,cs] fp32; block partial min/max (+ element index) for the global range normalise (slip.py:21-36)
void cutout_forward(const CutoutArgs& a, float* batch, float* part_min, float* part_max, int* part_imin,
                    int* part_imax, cudaStream_t st);
// multi-rank range exchange helpers: xbuf = {min, -max} for one allreduce(min)
void range_pack(const float* range, float* xbuf, cudaStream_t st);
void range_unpack(const float* xbuf, float* range, int* irange, cudaStream_t st);
// partials of an arbitrary buffer (same layout as cutout_forward's), nparts blocks
void minmax_partials(const float* x, long long n, int nparts, float* part_min, float* part_max, int* part_imin,
                     int* part_imax, cudaStream_t st);
// range[0]=min, range[1]=R (max of x-min, 1 if zero), range[2]=max, range[3]=R!=0; irange = argmin / argmax element
void minmax_reduce(const float* batch_or_null, const float* part_min, const float* part_max, const int* part_imin,
                   const int* part_imax, int nparts, float* range, int* irange, cudaStream_t st);
// patches[(n*gp + py)*gp + px, (c*P + iy)*P + ix] = ((x - min)/R - mean_c)/std_c   (slip.py:52-60 + conv1 im2col)
void patchify_forward(const float* batch, const float* range, int n, int cs, int P, int ld, act_t* patches,
                      cudaStream_t st);
// g_batch (=|+=) d/d(batch) of the direct term; sums_fx[0] += sum g_a, sums_fx[1] += sum g_a * a / R in 64-bit fixed point
// (order-independent: identical bits on every run); range_sums_finish converts to fp32 and clears the accumulator
void patchify_backward(const act_t* g_patches, const float* batch, const float* range, int n, int cs, int P, int ld,
                       int accumulate, float* g_batch, long long* sums_fx, FxPass fx, cudaStream_t st);
void range_sums_finish(long long* sums_fx, FxPass fx, float* sums, cudaStream_t st);
// adds the argmin / argmax terms of the global range normalise, then scatters through the bilinear taps
// g_pooled: [3, src_h, src_w] (overwritten); acc: zeroed fixed-point accumulator of the same extent (cleared again on return)
void cutout_backward(const CutoutArgs& a, const float* g_batch, const float* range, const int* irange,
                     const float* sums, long long* acc, FxPass fx, float* g_pooled, cudaStream_t st);

// ------------------------------------------------------------------ CLIP ViT (slip.py:62-66; SLIP/models.py:18-64)
// y = LN(x [+ pos[row % T]]) * gamma + beta ; x fp32 [rows, W]; outputs optional fp16 / fp32; stats [rows][2]
// W in {128, 256, 512, 768, 1024}; row r of x starts at x + r * x_stride (class-token rows: stride T * W)
void layernorm_forward(const float* x, long long x_stride, const float* pos, int T, const float* gamma,
                       const float* beta, int rows, int W, float eps, act_t* y16, float* y32, float* stats,
                       cudaStream_t st);
// the same on an fp16 residual stream (x fp16)
void layernorm_forward(const act_t* x, long long x_stride, const float* pos, int T, const float* gamma,
                       const float* beta, int rows, int W, float eps, act_t* y16, float* y32, float* stats,
                       cudaStream_t st);
// gx (+)= LN'(x) applied to dy (fp16, scaled); also writes gx16 = fp16(gx).  accumulate=0 overwrites gx.
// dy is compact [rows, W]; x, gx, gx16 rows are x_stride apart
void layernorm_backward(const act_t* dy, const float* x, long long x_stride, const float* pos, int T,
                        const float* stats, const float* gamma, int rows, int W, int accumulate, float* gx,
                        act_t* gx16, cudaStream_t st);
// fp16 residual stream: x fp16; with gx == nullptr the stream gradient lives in gx16 alone (accumulate reads it there)
void layernorm_backward(const act_t* dy, const act_t* x, long long x_stride, const float* pos, int T,
                        const float* stats, const float* gamma, int rows, int W, int accumulate, float* gx,
                        act_t* gx16, cudaStream_t st);
// in-place row softmax over the first `cols` of each row of length ld (pad columns zeroed); rows total
void softmax_forward(act_t* s, int rows, int cols, int ld, cudaStream_t st);
void softmax_backward(const act_t* p, act_t* dp_to_ds, int rows, int cols, int ld, cudaStream_t st);
// Prompt.forward for all prompts of one perceptor + its gradient w.r.t. the un-normalised embeds.
//   e [B, D]; prompts [n, D] (unit rows), weights/stops [n]; de [B, D].  slots / inv_rows (nullable): row j adds into
//   losses[slots[j]] with 1 / (rows of its Prompt) -- multi-row embeds (image prompts).  losses += partial, caller zeroes.
void prompt_loss(const float* e, int B, int D, const float* prompts, const float* weights, const float* stops,
                 const int* slots, const float* inv_rows, int n, int cutn_global, float grad_scale, float* e_unit,
                 float* losses, float* de, act_t* de16, cudaStream_t st);

// ------------------------------------------------------------------ optimiser (pixray.py:520-555, 1484-1487)
// The optimisers rebuild_optimisers can build (`--optimiser`), with the library defaults (the reference passes only lr):
// torch.optim.Adam, AdamW (weight decay 0.01), Adagrad (eps 1e-10, lr_decay 0, initial accumulator 0), Adamax, and
// torch_optimizer.DiffGrad 0.1.0.  Betas / eps of the Adam family come from pxr_config (defaults 0.9 / 0.999 / 1e-8).
// Values are the PXR_OPT_* of the C ABI.
enum OptKind { OPT_ADAM = 0, OPT_ADAMW = 1, OPT_ADAGRAD = 2, OPT_ADAMAX = 3, OPT_DIFFGRAD = 4 };
constexpr int OPT_KINDS = 5;
constexpr float ADAMW_WEIGHT_DECAY = 0.01f;
// Per-element state, z_numel floats each.  s0: first moment (Adam, AdamW, Adamax, DiffGrad); s1: second moment (Adam,
// AdamW, DiffGrad), sum of squared gradients (Adagrad) or infinity norm (Adamax); s2: previous gradient (DiffGrad).
struct OptState {
  float *s0, *s1, *s2;
};
// The step's scalars, from the learning rate and the step count t of the current optimiser instance (1-based).
struct OptCoef {
  float step_size;     // Adam / AdamW / Adamax: lr / (1 - b1^t); Adagrad: lr; DiffGrad: lr sqrt(1 - b2^t) / (1 - b1^t)
  float inv_sqrt_bc2;  // Adam / AdamW: 1 / sqrt(1 - b2^t)
  float decay;         // AdamW: 1 - lr * weight_decay, applied to z before the step
};
__host__ __device__ inline OptCoef opt_coef(int kind, float lr, float b1, float b2, int t) {
  const double bc1 = 1.0 - pow((double)b1, (double)t), bc2 = 1.0 - pow((double)b2, (double)t);
  OptCoef c;
  c.step_size = (float)((double)lr / bc1);
  c.inv_sqrt_bc2 = (float)(1.0 / sqrt(bc2));
  c.decay = kind == OPT_ADAMW ? (float)(1.0 - (double)lr * (double)ADAMW_WEIGHT_DECAY) : 1.f;
  if (kind == OPT_ADAGRAD) c.step_size = lr;
  if (kind == OPT_DIFFGRAD) c.step_size = (float)((double)lr * sqrt(bc2) / bc1);
  return c;
}
// One step of optimiser `kind` on z with gradient g * inv_scale (t = its step count, 1-based), then clip_z to
// per-channel [zmin, zmax] (vqgan.py:202-204) or [0,1] when zmin == nullptr && clip01.
void opt_clip_step(int kind, float* z, OptState s, const float* g, float inv_scale, int n, int per_channel,
                   const float* zmin, const float* zmax, int clip01, float lr, float b1, float b2, float eps, int t,
                   cudaStream_t st);

// ------------------------------------------------------------------ device-side checkdrop + optimiser step (pixray.py:1090-1109, 1464-1512)
// train()'s per-iteration control decisions without a host round trip.  The optimiser step of iteration `it` reads the
// iteration's loss vector, decides like checkdrop / the scheduled learning-rate drops / auto_stop do, applies the step +
// clip_z with the CURRENT learning rate and optimiser state, and -- when the decision is "rebuild the optimisers" --
// leaves a fresh optimiser of the same kind (state zeroed, t = 0) at learning_rate / 10^num_loss_drop behind for the next
// iteration, or raises `stopped` when the drops are used up (after which further iterations leave z untouched).  State
// is double-buffered (read cur, write next) so every block of the kernel sees the same decision inputs.
struct DropState {
  float best_loss;     // 1e20 after a rebuild (pixray.py:1509)
  int best_iter;
  int num_loss_drop;
  int stopped;
  float lr;
  int adam_t;          // steps taken by the current optimiser instance (whichever kind)
  int pad[2];
};
struct DropConfig {
  float base_lr;       // args.learning_rate, or the drawer's own rate (fftdrawer.py:63-67)
  int iter_drop_delay; // 12 (pixray.py:1987)
  int max_loss_drops;  // len(args.learning_rate_drops)
  int auto_stop;
  int n_sched;
  int sched[16];       // args.learning_rate_drops: iterations at which the rate drops regardless of the losses
};
// What the host may poll without synchronising (pinned, mapped memory; seq_begin == seq_end == iteration + 1 when the
// record is consistent).
struct DropStatus {
  volatile int seq_begin;
  int iter;
  float loss_sum, best_loss;
  int best_iter, num_loss_drop, stopped, rebuilt;
  float lr;
  int n_losses;
  float losses[64];
  volatile int seq_end;
};
void opt_clip_managed(int kind, float* z, OptState s, const float* g, float* best_z, float inv_scale, int n,
                      int per_channel, const float* zmin, const float* zmax, int clip01, float b1, float b2, float eps,
                      const float* losses, int n_losses, int iter, const DropConfig& cfg, const DropState* cur,
                      DropState* next, DropStatus* status_mapped, cudaStream_t st);
// acc (=|+=) g: gradient accumulation over the `batches` passes of one iteration (pixray.py:1464-1482)
void accumulate_f32(const float* g, float* acc, long long n, int accumulate, cudaStream_t st);

// ------------------------------------------------------------------ auxiliary losses (Losses/*.py), kernels_losses.cu
// Every launcher adds grad_scale * weight * dL/dx into the fp32 gradient buffer of the tensor the reference loss reads
// and writes (image losses) or accumulates (cutout / embedding losses: per-rank partial sums) the weighted loss value.
// `part`: scratch of max(4 * AUX_MAX_BLOCKS, n_local) doubles.  `weight` = the loss's own *_weight setting times the
// custom_loss spec weight (pixray.py:1388).
constexpr int AUX_MAX_BLOCKS = 1024;
// Anchors to a stored copy (pixray.py:1344-1375).  anchor_z: kind 0 spherical / 1 mse/2 / 2 cosine embedding between the
// latent and `ref` (n floats each), adds weight * dL/dz into z_grad (unscaled fp32) and writes the weighted value.
// anchor_pix: weight/2 * l1(img, ref) with its sign gradient (times grad_scale) into g_img.
void anchor_z(int kind, const float* z, const float* ref, int n, float weight, float* z_grad, float* loss_out, cudaStream_t st);
void anchor_pix(const float* img, const float* ref, long long n, float weight, float grad_scale, float* g_img, double* part,
                float* loss_out, cudaStream_t st);
void aux_symmetry(const float* img, int H, int W, float weight, float grad_scale, float* g_img, double* part,
                  float* loss_out, cudaStream_t st);
// margins = (left, right, upper, lower) in pixels (EdgeLoss.py:82-88), colour in [0,1]
void aux_edge(const float* img, int H, int W, const int margins[4], const float color[3], float edge_color_weight,
              float global_color_weight, float weight, float grad_scale, float* g_img, double* part, float* loss_out,
              cudaStream_t st);
void aux_gaussian(const float* img, int H, int W, float stdy, float stdx, const float color255[3], float weight,
                  float grad_scale, float* g_img, double* part, float* loss_out, cudaStream_t st);
// best_out (optional): nearest-palette index per pixel [n_img * cs * cs] (the loss's integer bookkeeping)
void aux_palette(const float* batch, int n_img, int cs, int cutn_global, const float* palette_dev, int n_colors,
                 float weight, float grad_scale, float* g_batch, int* best_out, double* part, float* loss_out,
                 cudaStream_t st);
// saturation: local moment sums (4 doubles) -> [allreduce over ranks] -> gradient from the global moments
void aux_saturation_moments(const float* batch, int n_img, int cs, double* part, double* sums, cudaStream_t st);
void aux_saturation_grad(const float* batch, int n_img, int cs, int cutn_global, const double* sums, float weight,
                         float grad_scale, int write_loss, float* g_batch, float* loss_out, cudaStream_t st);
// A: scratch [(n_img * cs + 2) * cs] floats; halo: [2][2][3][cs] rows around this rank's slab (unused when world == 1)
void aux_smoothness(const float* batch, int n_img, int cs, int first_global, int cutn_global, const float* halo,
                    float spacing, int kind, float weight, float grad_scale, float* A, float* g_batch, double* part,
                    float* loss_out, cudaStream_t st);
void aux_smooth_pack_halo(const float* batch, int n_img, int cs, int rank, float* xbuf, cudaStream_t st);
void aux_smooth_unpack_halo(const float* xbuf, int cs, int rank, int world, float* halo, cudaStream_t st);
void aux_aesthetic(const float* e, int n_local, int D, int cutn_global, const float* w_dev, float bias, float target,
                   float weight, float grad_scale, float* de, __half* de16, double* part, float* loss_out,
                   cudaStream_t st);

// ------------------------------------------------------------------ filters (kernels_filters.cu; filters/*.py, pixray.py:1203-1222)
// planar fp32 [3, H, W]; roll = torch.roll(x, (sh, sw), (2, 3)); *_backward: gx (=|+=) adjoint(gy)
void filter_roll(const float* x, int H, int W, int sh, int sw, float* y, cudaStream_t st);
void filter_roll_backward(const float* gy, int H, int W, int sh, int sw, int accumulate, float* gx, cudaStream_t st);
// wallpaper "shift": [3,H,W] -> [3,2H,W] (second row of tiles offset by W/2), rolled by (sh, sw)
void filter_wallpaper_shift(const float* x, int H, int W, int sh, int sw, float* y, cudaStream_t st);
void filter_wallpaper_shift_backward(const float* gy, int H, int W, int sh, int sw, int accumulate, float* gx, cudaStream_t st);
void filter_crop(const float* x, int H, int W, int top, int left, int Hc, int Wc, float* y, cudaStream_t st);
void filter_crop_backward(const float* gy, int H, int W, int top, int left, int Hc, int Wc, float* gx, cudaStream_t st);
// loss = weight * mse(first em, last em) / em along axis (0: columns, 1: rows); g (nullable) += grad_scale * dloss/dx
void filter_edge_match(const float* x, int H, int W, int em, int axis, float weight, float grad_scale, int accumulate_loss,
                       float* g, float* loss_out, cudaStream_t st);
// nearest palette colour (first minimum), loss = weight * (beta + 1) * mean((z_q - z)^2); part: AUX_MAX_BLOCKS doubles
void filter_colorlookup(const float* x, int pixels, const float* pal, int n_col, float beta, float weight, float* y,
                        int* best_out, double* part, float* loss_out, cudaStream_t st);
void filter_colorlookup_backward(const float* gy, const float* x, const float* y, int pixels, float beta, float weight,
                                 float grad_scale, int accumulate, float* gx, cudaStream_t st);

// ------------------------------------------------------------------ vdiff drawer (kernels_vdiff.cu; cc12m_1.py, sampling.py)
struct VdFeatures {
  float v[144];  // [cos, sin] Fourier features of t: 128 for the mapping network, 16 timestep planes
};
void vd_set_features(const VdFeatures& f, float* h0_tail, float* te, cudaStream_t st);
void vd_input(const float* x, const float* te, int pixels, act_t* out, cudaStream_t st);  // [pixels, 64]: x | te | 0
void avgpool2x(const act_t* x, int H, int W, int C, int ld_in, act_t* y, cudaStream_t st);
void avgpool2x_backward(const act_t* gy, int H, int W, int C, int accumulate, act_t* gx, cudaStream_t st);
void bilinear_up2x(const act_t* x, int H, int W, int C, act_t* y, int ld_out, cudaStream_t st);   // align_corners=False
void bilinear_up2x_backward(const act_t* gy, int H, int W, int C, int ld_gy, act_t* gx, cudaStream_t st);
void copy_channels(const act_t* src, int ld_src, act_t* dst, int ld_dst, int C, long long pixels, int accumulate,
                   cudaStream_t st);
void im2col3x3(const act_t* x, int H, int W, int C, act_t* A, cudaStream_t st);  // A [pixels, 9 C], tap-major
void gemv_f16(const act_t* W, int K, int R, const float* x, const float* bias, int relu, const float* res, float* y,
              cudaStream_t st);
void vd_finish(const float* vout, int ld, const float* x, float alpha, float sigma, int pixels, float* v_planar,
               float* pred, float* pre, float* img, cudaStream_t st);
void vd_finish_backward(const float* g_img, const float* pre, float sigma, int pixels, int ld, float* g_pred, act_t* g_v,
                        cudaStream_t st);
void vd_zgrad(const float* g_pred, const act_t* g_in, int ld, float alpha, float inv_scale, int pixels, float* z_grad,
              cudaStream_t st);
void vd_renoise(float* x, const float* pred, const float* v, const float* noise, float alpha_i, float sigma_i,
                float alpha_next, float adjusted_sigma, float ddim_sigma, long long n, cudaStream_t st);

void fill_f32(float* p, float v, long long n, cudaStream_t st);
void cast_f32_to_f16(const float* x, act_t* y, long long n, float scale, cudaStream_t st);

}  // namespace pxr
