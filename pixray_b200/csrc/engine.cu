// The engine behind include/pixray_b200.h: owns weights (repacked to the kernels' layouts), every activation /
// gradient buffer, the pre-built kernel plans ("op lists") for forward and the hand-written backward chain, Adam state
// and the per-iteration cutout parameters.  One handle = one rank = one CUDA stream.
//
// Hot path order per iteration (pixray.py:1243-1406, 1436-1512):
//   drawer.synth -> pool -> cutouts -> [per perceptor: patchify -> ViT -> head -> Prompt loss]
//   -> backward of all of the above by hand (dgrad only: every network is frozen, vqgan.py:125, slip.py:176)
//   -> [allreduce z.grad] -> Adam -> clip_z
#include "engine.cuh"
#include "comm.cuh"
#include "attn_tc.cuh"
#include "transforms.h"
#include <algorithm>
#include <atomic>
#include <map>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <memory>

namespace pxr {

static inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

struct VSpec;  // one element of the vdiff U-Net description (engine_vdiff.inc)

// ===================================================================================================== Engine
class Engine {
 public:
  pxr_config cfg;
  cudaStream_t st = nullptr;
  std::string err;
  int64_t launches = 0;
  int num_sms = 148;
  int fmt = 0;
  float S = 4096.f;  // grad scale
  bool fuse_softmax = false;  // PXR_FUSE_SOFTMAX=1: attention softmax inside the GEMM epilogue (see DESIGN.md 4)
  bool gn_coop = true;        // PXR_GN_COOP=0: three-kernel GroupNorm instead of the cooperative single-kernel one
  bool stream16 = true;       // the ViT residual stream and its gradient in fp16, like the reference's CUDA path (clip.load gives a half model, slip.py:176); PXR_CLIP_STREAM=32 keeps them in fp32
  bool fused_attn = true;     // PXR_FUSED_ATTN=0: fall back to the batched-GEMM attention (attn_tc.cu covers T <= 256)
  std::map<std::string, HostWeight> weights[3];
  std::vector<void*> allocs;
  bool finalized = false;
  std::map<std::string, std::pair<void*, size_t>> dbg;  // named internal buffers (tests / debugging)
  void reg(const std::string& n, void* p, size_t bytes) { dbg[n] = {p, bytes}; }

  // sharding
  int n_local = 0, first_global = 0;

  // ---- drawer
  float* z_buf = nullptr;   // engine copy of z
  float* z_grad = nullptr;
  float *adam_m = nullptr, *adam_v = nullptr;  // optimiser state s0 / s1 (kernels.cuh OptState)
  float* opt_prev = nullptr;                   // s2: DiffGrad's previous gradient
  int opt_kind = OPT_ADAM;                     // PXR_OPT_*
  int adam_t = 0;                              // steps of the current optimiser instance
  // device-side checkdrop / learning-rate drops / auto-stop (kernels.cuh): off until pxr_set_schedule
  bool managed = false;
  DropConfig drop_cfg{};
  DropState* drop_state = nullptr;        // [2], double-buffered on the device
  DropStatus* drop_status = nullptr;      // pinned, mapped
  DropStatus* drop_status_dev = nullptr;  // its device address
  float* best_z = nullptr;
  int drop_parity = 0;
  // gradient accumulation over the `batches` passes of one iteration (pixray.py:1464-1482)
  int batches = 1;
  float* z_grad_acc = nullptr;
  int rng_iter = 0;  // key of the engine-drawn cutout parameters: iteration, and pass within the iteration
  int64_t z_numel = 0;
  float *zmin = nullptr, *zmax = nullptr;  // [z_channels]
  float *img = nullptr, *img_pre = nullptr, *g_img = nullptr;  // [3,H,W]
  OpList drawer_fwd, drawer_bwd;  // bwd stored in execution order

  // ---- filters between synth and cutouts (do_synth_and_filter, pixray.py:1203-1222; filters/*.py), fused path only.
  // A filter is a short chain of primitives; `cut_img` / `g_cut_img` [3, cut_h, cut_w] are what MakeCutouts and the image
  // losses see (== img / g_img without filters; wallpaper "shift" doubles the height, edge_match trims).
  enum { FP_ROLL = 0, FP_WSHIFT = 1, FP_CROP = 2, FP_EDGE = 3, FP_LOOKUP = 4 };
  struct FilterPrim {
    int kind, filter;       // primitive kind, index of the filter it belongs to (= its loss slot)
    int Hin, Win, Hout, Wout;
    int use_h = 0, use_w = 0;            // ROLL: which shifts apply
    int top = 0, left = 0;               // CROP
    int em = 0, axis = 0, accumulate = 0;  // EDGE
    float beta = 0.f;                    // LOOKUP
    const float* in = nullptr;           // input tensor (forward)
    float* g_in = nullptr;               // gradient buffer of the input tensor
    float *out = nullptr, *g_out = nullptr;
  };
  struct Filter {
    int kind;               // PXR_FILTER_*
    float weight;
    int wp_type = 0, em = 0;
    float beta = 10.f;
    float* pal = nullptr;
    int n_col = 0;
    int H = 0, W = 0;       // input size of the filter (the shifts are drawn in [0, H) x [0, W), like the reference)
    int sh = 0, sw = 0;     // this iteration's shifts
    int fixed_h = -1, fixed_w = -1;  // explicit shifts for replays (pxr_set_filter_shifts)
  };
  std::vector<Filter> filters;
  std::vector<FilterPrim> fprims;
  float *cut_img = nullptr, *g_cut_img = nullptr;
  int cut_h = 0, cut_w = 0;
  bool filtered_valid = false;  // cut_img holds the filtered image of the current z (fused path); else use img
  float* filter_dummy = nullptr;
  int* lookup_best = nullptr;
  void rebuild_filters();
  void filters_forward(int iter);
  void filters_backward();
  const float* cur_cut_img() const { return filtered_valid ? cut_img : img; }
  float* cur_g_cut_img() const { return filtered_valid ? g_cut_img : g_img; }
  int cur_cut_h() const { return filtered_valid ? cut_h : cfg.image_h; }
  int cur_cut_w() const { return filtered_valid ? cut_w : cfg.image_w; }

  // ---- cutouts
  float *pooled = nullptr, *g_pooled = nullptr, *batch = nullptr, *g_batch = nullptr;
  // non-square canvas (cfg.cut_aspect != 1): the warps sample from a stretch of the pooled image (pixray.py:468-472)
  double aspect = 1.0;
  int src_h = 0, src_w = 0;
  float *cut_src = nullptr, *g_cut_src = nullptr;  // [3, src_h, src_w]; == pooled / g_pooled when square
  int* pool_argmax = nullptr;
  float *part_min = nullptr, *part_max = nullptr, *range = nullptr, *sums = nullptr;
  long long *sums_fx = nullptr, *grad_fx = nullptr;  // 64-bit fixed-point accumulators (order-independent sums, kernels_cutouts.cu)
  unsigned int* fx_poison = nullptr;                   // [2]: pass id of the last non-finite contribution to {gradient images, range sums}
  unsigned int fx_pass = 0;
  FxPass next_fx(int word) {
    FxPass f;
    f.poison = fx_poison + word;
    f.pass = ++fx_pass;
    return f;
  }
  int *part_imin = nullptr, *part_imax = nullptr, *irange = nullptr;
  int n_parts = 0;
  static constexpr int RING = 8;
  float* minv_host[RING] = {nullptr};   // pinned
  float* facs_host[RING] = {nullptr};
  cudaEvent_t ring_ev[RING] = {nullptr};
  int ring_pos = 0;
  float *minv_dev = nullptr, *facs_dev = nullptr;
  float cj_p = 0.8f, cj_sat = 0.1f, cj_hue = 0.1f;  // K.ColorJitter(hue=0.1, saturation=0.1, p=0.8), pixray.py:416, 436
  CutoutArgs cut_args;

  // ---- perceptors
  struct Clip {
    pxr_clip_cfg c;
    int T, np, Kp, ldT, M, B;
    // weights
    act_t* conv1 = nullptr;
    float *cls = nullptr, *pos = nullptr, *proj = nullptr;
    NormW ln_pre, ln_post;
    struct Layer {
      act_t *wqkv, *wo, *wfc, *wproj;
      float *bqkv, *bo, *bfc, *bproj;
      NormW ln1, ln2;
      // saved activations
      void *x_in, *x_mid;  // residual stream before / between the two sub-blocks: fp32, or fp16 with stream16
      float *stats1, *stats2;
      act_t *qkv, *P, *u;
      act_t* o = nullptr;     // fused attention: per-layer attention output (backward needs D = dO . O)
      float* lse = nullptr;   // fused attention: row log-sum-exp [B, heads, T]
      std::shared_ptr<AttnPlan> attn;
    };
    std::vector<Layer> layers;
    // buffers
    act_t *patches, *g_patches, *h16, *o16, *gact, *g4, *gh, *go, *gqkv, *dP, *gx16;
    float *t, *stats_pre, *stats_post, *e, *e_unit, *de, *gx;
    void* x_out;  // residual stream after the last block (fp32 / fp16)
    act_t *proj16, *hcls, *gcls, *de16;
    // prompts
    float *prompts = nullptr, *pweights = nullptr, *pstops = nullptr, *losses = nullptr;
    int n_prompts = 0, loss_offset = 0;  // n_prompts = loss slots of this perceptor (text + image prompts)
    // rows of `prompts`: n_text single-row Prompts, then cutn rows per image prompt (refreshed every iteration)
    std::vector<float> text_rows, text_w, text_stop;
    int n_text = 0, n_rows = 0;
    int* pslot = nullptr;
    float* pinv = nullptr;
    float* scratch = nullptr;  // pxr_prompt_loss on caller-provided embeddings
    // spot prompts (pixray.py:1283-1293): text Prompts scored on the embeddings of the masked cutouts.
    // [1] = args.spot_prompts (make_cutouts(out, spot=1)), [0] = args.spot_prompts_off (spot=0)
    struct Spot {
      std::vector<float> rows, w, stop;
      int n = 0, loss_offset = 0;
      float *d_rows = nullptr, *d_w = nullptr, *d_stop = nullptr, *d_inv = nullptr;
      int* d_slot = nullptr;
    } spot[2];
    OpList fwd, bwd;
  };
  Clip clip[2];
  float* losses_dev = nullptr;   // [total prompts]
  float* losses_scratch = nullptr;  // loss vector of the passes b > 0 of an iteration (batches > 1)
  float* losses_host = nullptr;  // pinned
  int total_prompts = 0;
  // image prompts (pixray.py:1308-1336): target images, cut + encoded every iteration with the cached transforms
  float* img_prompts = nullptr;  // [n_img, 3, cs, cs]: the POOLED targets ((avg + max) / 2 of each image at its own size,
                                 // pixray.py:463): constants, pooled once when they are set, not every iteration
  int n_img = 0;
  std::vector<float> img_w;
  void rebuild_prompt_rows();
  void encode_image_prompts();
  // spot passes: the mask (device [3, cs, cs], != 0 where the mask image is >= 0.5) and the masked pooled image
  unsigned char* spot_mask = nullptr;
  float* pooled_masked = nullptr;
  bool any_spot(int which) const {
    for (int i = 0; i < cfg.n_clip; ++i)
      if (clip[i].spot[which].n > 0) return true;
    return false;
  }
  bool spot_accumulated = false;  // a spot pass of this iteration already wrote d loss / d image: the main pass adds to it
  bool spot_pass(int which, bool accumulate_img);
  void backward_to_image(const CutoutArgs& a, int mask_which, bool accumulate_img, bool main_pass);
  void backward_drawer();

  // ---- auxiliary losses (Losses/*.py; pixray.py:1384-1393): extra loss-vector entries after the prompts
  struct AuxLoss {
    int kind;
    float weight;
    std::vector<float> prm;
    float* dev = nullptr;  // palette colours / aesthetic head weights
    int n_dev = 0;
  };
  std::vector<AuxLoss> aux;
  double* aux_part = nullptr;   // reduction scratch
  double* aux_sums = nullptr;   // saturation moments (4)
  float* aux_A = nullptr;       // smoothness per-pixel factor
  float* aux_halo = nullptr;    // smoothness rows of the neighbouring ranks
  float* aux_xbuf = nullptr;    // smoothness halo exchange buffer
  int* aux_best = nullptr;      // palette argmin per pixel (bookkeeping, also a debug buffer)
  // ---- anchors to a stored copy (pixray.py:1344-1375): loss-vector entries between the prompts and the auxiliary losses
  struct Anchor {
    int kind;      // PXR_ANCHOR_*
    float weight;
    float* ref = nullptr;
    size_t n = 0;
  };
  std::vector<Anchor> anchors;
  void anchors_on_image();  // init_weight_pix: into the (filtered) image gradient, before the drawer backward
  void anchors_on_z();      // z-space terms: into z.grad, after the drawer backward
  int aux_base() const { return total_prompts + (int)anchors.size(); }
  int num_losses() const { return aux_base() + (int)aux.size(); }  // total_prompts includes the filter slots in front
  void aux_after_embed();   // aesthetic: needs de of the last perceptor (after its prompt_loss)
  void aux_on_cutouts();    // saturation / palette / smoothness: add into g_batch
  void aux_on_image();      // symmetry / edge / gaussian: add into g_img

  // ---- comm (multi-GPU, cutout sharding): one NCCL communicator owned by the engine (comm.cuh)
  void* comm = nullptr;
  float* xbuf = nullptr;  // {min, -max} exchange buffer
  void nccl_check(int rc, const char* what) {
    if (rc != 0) {
      const char* m = Comm::api().err_str ? Comm::api().err_str(rc) : "?";
      throw EngineError(-91, std::string(what) + ": NCCL error " + m);
    }
  }

  explicit Engine(const pxr_config& c) : cfg(c) {}
  ~Engine();

  template <class T>
  T* dalloc(size_t n, bool zero = true) {
    void* p = nullptr;
    size_t bytes = (n * sizeof(T) + 255) / 256 * 256;
    PXR_CUDA(cudaMalloc(&p, bytes));
    if (zero) PXR_CUDA(cudaMemsetAsync(p, 0, bytes, st));
    allocs.push_back(p);
    return static_cast<T*>(p);
  }
  // release one tracked allocation early (buffers that are rebuilt when prompts change); cudaFree waits for the device
  template <class T>
  void dfree(T*& p) {
    if (!p) return;
    auto it = std::find(allocs.begin(), allocs.end(), static_cast<void*>(p));
    if (it != allocs.end()) {
      cudaFree(*it);
      allocs.erase(it);
    }
    p = nullptr;
  }
  template <class T>
  T* upload(const std::vector<T>& v) {
    T* p = dalloc<T>(v.size(), false);
    PXR_CUDA(cudaMemcpyAsync(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, st));
    PXR_CUDA(cudaStreamSynchronize(st));  // v may be a temporary
    return p;
  }
  act_t* upload_f16(const std::vector<float>& v) {
    std::vector<act_t> h(v.size());
    for (size_t i = 0; i < v.size(); ++i) h[i] = __float2half_rn(v[i]);
    return upload(h);
  }
  const HostWeight& W(int mod, const std::string& name, std::initializer_list<int64_t> dims = {}) {
    auto it = weights[mod].find(name);
    if (it == weights[mod].end()) throw EngineError(-40, "missing weight '" + name + "' (module " + std::to_string(mod) + ")");
    if (dims.size()) {
      std::vector<int64_t> want(dims);
      if (it->second.dims != want) {
        std::string got;
        for (auto d : it->second.dims) got += std::to_string(d) + ",";
        throw EngineError(-41, "weight '" + name + "' has shape [" + got + "] which does not match the configured architecture");
      }
    }
    return it->second;
  }

  // profiling (pxr_profile_iteration): CUDA-event pair around every op, split gemm_tc_kernel vs everything else
  bool profiling = false;
  struct ProfRec {
    cudaEvent_t a, b;
    double flops;
    double bytes;
    int launches;
    std::string name;
  };
  std::vector<ProfRec> prof;
  void prof_begin(ProfRec& r) {
    PXR_CUDA(cudaEventCreate(&r.a));
    PXR_CUDA(cudaEventCreate(&r.b));
    PXR_CUDA(cudaEventRecord(r.a, st));
  }
  bool trace = false;  // PXR_TRACE=1: print every op before it runs and synchronise after it (localises a hanging kernel)
  void run(OpList& l) {
    for (size_t i = 0; i < l.ops.size(); ++i) {
      if (trace) {
        fprintf(stderr, "[pxr op] %s\n", l.names[i].empty() ? "(unnamed)" : l.names[i].c_str());
        fflush(stderr);
        l.ops[i]();
        cudaError_t e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) throw EngineError(-202, std::string("op '") + l.names[i] + "' failed: " + cudaGetErrorString(e));
      } else if (profiling) {
        ProfRec r;
        r.flops = l.flops[i];
        r.bytes = l.bytes[i];
        r.launches = l.launches[i];
        r.name = l.names[i];
        prof_begin(r);
        l.ops[i]();
        PXR_CUDA(cudaEventRecord(r.b, st));
        prof.push_back(r);
      } else {
        l.ops[i]();
      }
      launches += l.launches[i];
    }
  }
  void check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) throw EngineError(-201, std::string(what) + ": " + cudaGetErrorString(e));
  }

  // ------------------------------------------------------------------ plan helpers
  static GemmOperand opK(const void* p, long long ld, long long mn, long long k, int nb0 = 1, long long bs0 = 0,
                         int nb1 = 1, long long bs1 = 0) {
    GemmOperand o;
    o.ptr = p;
    o.mode = OP_KMAJOR;
    o.ld = ld;
    o.mn_extent = mn;
    o.k_extent = k;
    o.nb0 = nb0;
    o.nb1 = nb1;
    o.bs0 = bs0;
    o.bs1 = bs1;
    return o;
  }
  static GemmOperand opMN(const void* p, long long ld, long long mn, long long k, int nb0 = 1, long long bs0 = 0,
                          int nb1 = 1, long long bs1 = 0) {
    GemmOperand o = opK(p, ld, mn, k, nb0, bs0, nb1, bs1);
    o.mode = OP_MNMAJOR;
    return o;
  }
  // Tile width by a wave-quantisation cost model: a persistent grid of num_sms CTAs runs ceil(tiles / num_sms) waves
  // of tiles whose cost grows with bn (plus a fixed per-tile overhead); e.g. M = 12608, N = 768 is 297 tiles of 256
  // (3 waves for 2.007 waves of work) but 396 tiles of 192 (3 cheaper waves).
  int pick_bn(int N, bool b_mn, long long m_tiles) const {
    const int step = b_mn ? 64 : 16;
    {  // PXR_GEMM_BN="3072:256,768:192": tile width by output width, for A/B measurements of the cost model's choices
      static const std::map<int, int> forced = [] {
        std::map<int, int> m;
        if (const char* e = getenv("PXR_GEMM_BN")) {
          int n = 0, bn = 0, used = 0;
          while (sscanf(e, "%d:%d%n", &n, &bn, &used) == 2) {
            m[n] = bn;
            e += used;
            if (*e == ',') ++e;
          }
        }
        return m;
      }();
      auto it = forced.find(N);
      if (it != forced.end() && it->second % step == 0 && m_tiles > 16) return it->second;
    }
    if (N <= 256 && m_tiles * 1 >= num_sms / 2) return round_up(N, step);
    int best = 0;
    double best_cost = 1e30;
    // CTA pairs (cta_group::2) schedule 256-row tile pairs over num_sms / 2 clusters
    const bool paired = m_tiles >= 2 && gemm_default_cta_group() == 2;
    const long long m_units = paired ? (m_tiles + 1) / 2 : m_tiles;
    const long long sm_units = paired ? num_sms / 2 : num_sms;
    for (int bn = 256; bn >= 64; bn -= 64) {
      if (bn % step) continue;
      if (paired && b_mn && bn % 128) continue;
      const long long tiles = m_units * ((N + bn - 1) / bn);
      const long long waves = (tiles + sm_units - 1) / sm_units;
      // narrower tiles re-read A more often and sit closer to the smem-bandwidth limit: mild penalty
      const double cost = (double)waves * (bn + 40.0) * (bn >= 192 ? 1.0 : (bn == 128 ? 1.06 : 1.2));
      if (cost < best_cost - 1e-9) {
        best_cost = cost;
        best = bn;
      }
    }
    if (N < best) best = round_up(N, step);
    return best;
  }
  void add_gemm(OpList& l, const GemmOperand& A, const GemmOperand& B, int M, int N, int K, const GemmEpilogue& e,
                int bn = 0) {
    if (!bn) bn = pick_bn(N, B.mode == OP_MNMAJOR, (long long)((M + 127) / 128) * A.nb0 * A.nb1);
    auto plan = std::make_shared<GemmPlan>();
    char buf[256] = {0};
    int rc = gemm_plan_make(plan.get(), A, B, M, N, K, e, bn, fmt, num_sms, buf, sizeof buf);
    if (rc) throw EngineError(rc, std::string("gemm plan: ") + buf);
    cudaStream_t s = st;
    l.add(1, [plan, s] { gemm_launch(*plan, s); }, plan->flops, gemm_label("gemm", *plan, A.mode, B.mode, e), plan->bytes);
  }
  static std::string gemm_label(const char* kind, const GemmPlan& p, int am, int bm, const GemmEpilogue& e) {
    char b[256];
    snprintf(b, sizeof b, "%s M=%d N=%d K=%d batch=%d bn=%d cg=%d A%s B%s act=%d%s%s%s%s%s%s", kind, p.p.M, p.p.N,
             p.p.num_k_blocks * GEMM_BLOCK_K, p.p.total_tiles / (p.p.tiles_m * p.p.tiles_n), p.p.block_n, p.p.cta_group, am == OP_MNMAJOR ? "mn" : "k", bm == OP_MNMAJOR ? "mn" : "k",
             e.act, e.bias ? " bias" : "", e.res_f32 ? " res32" : "", e.res_f16 ? " res16" : "", e.out_f32 ? " o32" : "",
             e.out_f16 ? " o16" : "", e.aux_out ? " aux" : "");
    return b;
  }
  // Small-spatial convolutions (16x16 / 32x32 latents: 2..64 output tiles, K up to 4608) leave most SMs idle and are
  // bound by the per-SM operand feed; split-K spreads the taps over the idle SMs (fp32 partial sums to a workspace, then
  // one fixed-order reduce + bias / residual / fp16 epilogue kernel: deterministic).
  bool conv_splitk = true;  // PXR_CONV_SPLITK=0 disables
  bool clip_last_cls = true;  // PXR_CLIP_LAST_CLS=0: the last ViT layer's row-wise tail on all rows instead of the class rows
  bool gn_group = true;     // PXR_GN_GROUP=0: never use the cluster-per-group GroupNorm (kernels_gn_group.cu)
  bool gn_fuse_sk = true;   // PXR_GN_FUSE_SPLITK=0: keep splitk_reduce and GroupNorm as two kernels
  bool gn_fuse_fwd = true, gn_fuse_bwd = true;  // PXR_GN_FUSE_FWD / PXR_GN_FUSE_BWD = 0: per direction (diagnostics)
  // the split-K reduce most recently appended by add_conv: a GroupNorm over exactly its output, appended next to the same
  // list, replaces that op by the fused reduce + GroupNorm kernel
  // (one slot per op list: forward and backward lists are built interleaved)
  struct PendingSplitK {
    size_t op_index = 0;
    const act_t* out = nullptr;
    int ld_out = 0, n_out = 0;
    long long px = 0;
    GnSplitK sk;
  };
  std::map<const OpList*, PendingSplitK> pend_sk;
  const GnSplitK* take_pending_splitk(OpList& l, const act_t* tensor, int px, int C, bool need_plain) {
    auto it = pend_sk.find(&l);
    if (!gn_fuse_sk || it == pend_sk.end()) return nullptr;
    const PendingSplitK& q = it->second;
    if (l.ops.empty() || q.op_index != l.ops.size() - 1 || q.out != tensor || q.px != px || q.n_out != C || q.ld_out != C)
      return nullptr;
    if (need_plain && (q.sk.bias || q.sk.res)) return nullptr;
    return &q.sk;
  }
  float* splitk_ws = nullptr;
  size_t splitk_ws_elems = 0;
  void add_conv(OpList& l, const act_t* in, int H, int Wd, int cin, const act_t* wt, int cout_pad, int n_out, int ks,
                const GemmEpilogue& e) {
    const long long m_tiles = (long long)(H * Wd + 127) / 128;
    int bn = pick_bn(cout_pad < 64 ? cout_pad : n_out, false, m_tiles);
    if (bn > cout_pad) bn = cout_pad;
    cudaStream_t s = st;
    char kind[32];
    snprintf(kind, sizeof kind, "conv%dx%d", ks, ks);
    const int nkb = ks * ks * cin / 64;
    const long long tiles = m_tiles * ((n_out + bn - 1) / bn);
    int splits = 1;
    if (conv_splitk && splitk_ws && e.out_f16 && !e.out_f32 && !e.res_f32 && !e.aux_out && e.act == ACT_NONE &&
        n_out % 8 == 0 && e.ldc % 8 == 0 && tiles * 2 <= num_sms && nkb >= 8) {
      const int want = (int)std::min<long long>(num_sms / tiles, nkb / 4);
      if (want >= 2) {
        const int kbps = (nkb + want - 1) / want;
        splits = (nkb + kbps - 1) / kbps;
      }
      if ((size_t)splits * H * Wd * n_out > splitk_ws_elems) splits = 1;
    }
    auto plan = std::make_shared<GemmPlan>();
    char buf[256] = {0};
    if (splits > 1) {
      GemmEpilogue pe;
      pe.out_f32 = splitk_ws;
      pe.ldc = n_out;
      pe.k_splits = splits;
      int rc = conv_plan_make(plan.get(), in, cin, 1, H, Wd, cin, wt, cout_pad, n_out, ks, pe, bn, fmt, num_sms, buf, sizeof buf);
      if (rc) throw EngineError(rc, std::string("conv plan (split-K): ") + buf);
      const float* ws = splitk_ws;
      const float* bias = e.bias;
      const act_t* res = e.res_f16;
      act_t* out = e.out_f16;
      const int ld_out = (int)e.ldc;
      const long long px = (long long)H * Wd;
      std::string label = gemm_label(kind, *plan, OP_KMAJOR, OP_KMAJOR, e) + " splitK=" + std::to_string(plan->p.k_splits);
      l.add(1, [=] { gemm_launch(*plan, s); }, plan->flops, label, plan->bytes);
      // the reduce is its own op so that a GroupNorm right behind it can absorb it (add_gn / add_gn_bwd)
      l.add(1, [=] { splitk_reduce(ws, plan->p.k_splits, px, n_out, n_out, bias, res, out, ld_out, s); }, 0.0,
            "splitk_reduce px=" + std::to_string(px) + " N=" + std::to_string(n_out) + " splits=" + std::to_string(plan->p.k_splits));
      PendingSplitK& q = pend_sk[&l];
      q.op_index = l.ops.size() - 1;
      q.out = out;
      q.ld_out = ld_out;
      q.px = px;
      q.n_out = n_out;
      q.sk.ws = ws;
      q.sk.splits = plan->p.k_splits;
      q.sk.ld_ws = n_out;
      q.sk.bias = bias;
      q.sk.res = res;
      q.sk.out = out;
      return;
    }
    int rc = conv_plan_make(plan.get(), in, cin, 1, H, Wd, cin, wt, cout_pad, n_out, ks, e, bn, fmt, num_sms, buf,
                            sizeof buf);
    if (rc) throw EngineError(rc, std::string("conv plan: ") + buf);
    l.add(1, [plan, s] { gemm_launch(*plan, s); }, plan->flops, gemm_label(kind, *plan, OP_KMAJOR, OP_KMAJOR, e), plan->bytes);
  }

  // Split-K for a plain K-major GEMM with few output tiles and a long reduction (the vdiff U-Net's 4x4 ... 1x1 levels:
  // M <= 16 pixels, K = 9 * cin up to 18432): partial sums to the shared workspace, then the same fixed-order reduce.
  void add_gemm_splitk(OpList& l, const GemmOperand& A, const GemmOperand& B, int M, int N, int K, const GemmEpilogue& e) {
    const int bn = pick_bn(N, false, (M + 127) / 128);
    const int nkb = (K + GEMM_BLOCK_K - 1) / GEMM_BLOCK_K;
    const long long tiles = (long long)((M + 127) / 128) * ((N + bn - 1) / bn);
    int splits = 1;
    if (conv_splitk && splitk_ws && e.out_f16 && !e.out_f32 && !e.res_f32 && !e.aux_out && e.act == ACT_NONE && e.alpha == 1.f &&
        N % 8 == 0 && e.ldc % 8 == 0 && tiles * 2 <= num_sms && nkb >= 8) {
      const int want = (int)std::min<long long>(num_sms / tiles, nkb / 4);
      if (want >= 2) {
        const int kbps = (nkb + want - 1) / want;
        splits = (nkb + kbps - 1) / kbps;
      }
      if ((size_t)splits * M * N > splitk_ws_elems) splits = 1;
    }
    if (splits <= 1) {
      add_gemm(l, A, B, M, N, K, e);
      return;
    }
    auto plan = std::make_shared<GemmPlan>();
    char buf[256] = {0};
    GemmEpilogue pe;
    pe.out_f32 = splitk_ws;
    pe.ldc = N;
    pe.k_splits = splits;
    pe.tma_epi = -1;
    int rc = gemm_plan_make(plan.get(), A, B, M, N, K, pe, bn, fmt, num_sms, buf, sizeof buf);
    if (rc) throw EngineError(rc, std::string("gemm plan (split-K): ") + buf);
    cudaStream_t s = st;
    const float* ws = splitk_ws;
    const float* bias = e.bias;
    const act_t* res = e.res_f16;
    act_t* out = e.out_f16;
    const int ld_out = (int)e.ldc;
    std::string label = gemm_label("gemm", *plan, A.mode, B.mode, e) + " splitK=" + std::to_string(plan->p.k_splits);
    l.add(2, [=] {
      gemm_launch(*plan, s);
      splitk_reduce(ws, plan->p.k_splits, M, N, N, bias, res, out, ld_out, s);
    }, plan->flops, label, plan->bytes);
  }

  // ------------------------------------------------------------------ build steps
  void create();
  void finalize();
  void build_vqgan();
  void build_pixel();
  void build_fft();
  FftPlans* fft = nullptr;
  void build_cutouts();
  void build_clip(int i);
  ConvW load_conv(const std::string& prefix, int cin, int cout, int ks, int cin_real = 0);
  // VQGAN encoder (taming Encoder + quant_conv + nearest code): VqganDrawer.init_from_tensor / reapply_from_tensor /
  // get_z_from_tensor (vqgan.py:174-185).  Forward only; built at finalize when the checkpoint carries encoder.* tensors.
  OpList enc_fwd;
  bool have_encoder = false;
  float* enc_img = nullptr;   // [3, H, W] input in [-1, 1]
  float* enc_z = nullptr;     // [C, hw] result
  void build_vqgan_encoder();
  NormW load_norm(int mod, const std::string& prefix, int c);
  Act new_act(int H, int Wd, int C) {
    Act a;
    a.H = H;
    a.W = Wd;
    a.C = C;
    a.p = dalloc<act_t>((size_t)H * Wd * C);
    a.g = dalloc<act_t>((size_t)H * Wd * C);
    return a;
  }
  // decoder blocks: append forward ops to drawer_fwd, push the backward closure list (reverse order) to bwd_stack
  std::vector<OpList> bwd_stack;
  float* gn_part = nullptr;  // scratch for GN partial sums (sized for the largest layer)
  GridBarrier gn_bar;        // grid barrier state of the single-kernel GroupNorm
  Act conv_fwd_bwd(const Act& x, const ConvW& w, OpList& bwd);
  Act resblock(const Act& x, const std::string& prefix, int cin, int cout);
  Act attnblock(const Act& x, const std::string& prefix, int c);
  Act upsample(const Act& x, const std::string& prefix);
  struct GNSaved {
    float* stats;
    float* gstats;
  };
  GNSaved add_gn(OpList& l, const Act& x, const NormW& n, int swish, act_t* y);
  void add_gn_bwd(OpList& l, const act_t* dy, const act_t* x, const GNSaved& s, const NormW& n, int px, int C, int swish,
                  const act_t* dres, act_t* dx);

  // ------------------------------------------------------------------ vdiff drawer (engine_vdiff.inc)
  struct VConv;
  void build_vdiff();
  VConv vd_load_conv(const std::string& prefix, int cin_real, int cin, int cout, int ks, bool has_bias, bool tiny);
  void vd_conv_fwd(OpList& l, const act_t* x, int H, int Wd, const VConv& v, GemmEpilogue e);
  void vd_conv_bwd(OpList& l, const act_t* dy, int H, int Wd, const VConv& v, GemmEpilogue e);
  GNSaved vd_norm(OpList& l, const Act& x, const float* gamma, const float* beta, float gamma_add, int act,
                  const act_t* res, act_t* y);
  void vd_norm_bwd(OpList& l, const act_t* dy, const Act& x, const GNSaved& s, const float* gamma, const float* beta,
                   float gamma_add, int act, const act_t* dres, act_t* dx);
  Act vd_block(const Act& x, const std::string& key, const VSpec& sp);
  Act vd_attn(const Act& x, const std::string& key, const VSpec& sp);
  Act vd_skip(const Act& x, const std::string& key, const VSpec& sp);
  Act vd_elem(const Act& x, const std::string& key, const VSpec& sp);
  int vd_add_modulation(const std::string& wkey, int c);
  void vdiff_prepare(int iter);
  void vdiff_forward();
  void vdiff_backward();
  std::vector<float> vd_steps, vd_alphas, vd_sigmas, vd_map_ff, vd_t_ff, vd_mod_host;
  bool vd_have_embed = false;
  int vd_iter = 0, vd_iter_request = 0, vd_mod_rows = 0;
  float *vd_pred = nullptr, *vd_v = nullptr, *vd_gpred = nullptr, *vd_vout = nullptr, *vd_mod_out = nullptr,
        *vd_h0 = nullptr, *vd_te = nullptr, *vd_tmp[5] = {nullptr}, *vd_b[5] = {nullptr};
  act_t *vd_gv = nullptr, *vd_col = nullptr, *vd_xin = nullptr, *vd_gin = nullptr, *vd_wmod = nullptr, *vd_w[5] = {nullptr};

  // ------------------------------------------------------------------ execution
  void prepare_cut_params(const pxr_cut_params* p, int iter);
  void forward_drawer() {
    if (cfg.drawer == PXR_DRAWER_VDIFF) vdiff_forward();
    else run(drawer_fwd);
  }
  void forward_cutouts();
  void forward_clip(int i);
  void loss_clip(int i);
  void backward_all();
  void step(float lr);
  void step_managed(int iter);
  void write_initial_drop_state();
  void zero_optimizer_state();
};

Engine::~Engine() {
  if (st) cudaStreamSynchronize(st);
  if (comm && Comm::api().destroy) Comm::api().destroy(comm);
  fft_plans_destroy(fft);
  for (void* p : allocs) cudaFree(p);
  for (int i = 0; i < RING; ++i) {
    if (minv_host[i]) cudaFreeHost(minv_host[i]);
    if (facs_host[i]) cudaFreeHost(facs_host[i]);
    if (ring_ev[i]) cudaEventDestroy(ring_ev[i]);
  }
  if (losses_host) cudaFreeHost(losses_host);
  if (drop_status) cudaFreeHost(const_cast<DropStatus*>(drop_status));
  if (st) cudaStreamDestroy(st);
}

void Engine::create() {
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    throw EngineError(-1, "no CUDA device: pixray_b200 has no CPU fallback");
  if (cfg.device < 0 || cfg.device >= ndev) throw EngineError(-2, "invalid CUDA device ordinal");
  PXR_CUDA(cudaSetDevice(cfg.device));
  cudaDeviceProp prop;
  PXR_CUDA(cudaGetDeviceProperties(&prop, cfg.device));
  if (prop.major != 10) throw EngineError(-3, std::string("pixray_b200 needs an sm_100 GPU (B200); found ") + prop.name);
  num_sms = prop.multiProcessorCount;
  PXR_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
  if (cfg.world < 1) cfg.world = 1;
  if (cfg.cutn % cfg.world) throw EngineError(-4, "cutn must be divisible by world");
  n_local = cfg.cutn / cfg.world;
  first_global = cfg.rank * n_local;
  fmt = cfg.op_dtype;
  if (fmt != PXR_DTYPE_F16) throw EngineError(-5, "only PXR_DTYPE_F16 operands are wired through the pointwise kernels");
  if (cfg.grad_scale > 0) S = cfg.grad_scale;
  if (const char* fs = getenv("PXR_FUSE_SOFTMAX")) fuse_softmax = atoi(fs) != 0;
  if (const char* fa = getenv("PXR_FUSED_ATTN")) fused_attn = atoi(fa) != 0;
  if (const char* cs16 = getenv("PXR_CLIP_STREAM")) stream16 = atoi(cs16) != 32;
  if (const char* gc = getenv("PXR_GN_COOP")) gn_coop = atoi(gc) != 0;
  if (const char* sk = getenv("PXR_CONV_SPLITK")) conv_splitk = atoi(sk) != 0;
  if (const char* lc = getenv("PXR_CLIP_LAST_CLS")) clip_last_cls = atoi(lc) != 0;
  if (const char* gg = getenv("PXR_GN_GROUP")) gn_group = atoi(gg) != 0;
  if (const char* gf = getenv("PXR_GN_FUSE_SPLITK")) gn_fuse_sk = atoi(gf) != 0;
  if (const char* gf = getenv("PXR_GN_FUSE_FWD")) gn_fuse_fwd = atoi(gf) != 0;
  if (const char* gf = getenv("PXR_GN_FUSE_BWD")) gn_fuse_bwd = atoi(gf) != 0;
  if (const char* tr = getenv("PXR_TRACE")) trace = atoi(tr) != 0;
  if (cfg.beta1 <= 0) cfg.beta1 = 0.9f;
  if (cfg.beta2 <= 0) cfg.beta2 = 0.999f;
  if (cfg.adam_eps <= 0) cfg.adam_eps = 1e-8f;
  if (cfg.cut_size % 4) throw EngineError(-6, "cut_size must be a multiple of 4");
}

// ===================================================================================================== weights
NormW Engine::load_norm(int mod, const std::string& prefix, int c) {
  NormW n;
  n.gamma = upload(W(mod, prefix + ".weight", {c}).data);
  n.beta = upload(W(mod, prefix + ".bias", {c}).data);
  return n;
}

// cin_real < cin: the stored tensor has cin_real input channels and the activation is zero-padded to cin (conv_in: 3 -> 64)
ConvW Engine::load_conv(const std::string& prefix, int cin, int cout, int ks, int cin_real) {
  if (cin_real <= 0) cin_real = cin;
  const HostWeight& w = W(PXR_MOD_VQGAN, prefix + ".weight", {cout, cin_real, ks, ks});
  const HostWeight& b = W(PXR_MOD_VQGAN, prefix + ".bias", {cout});
  ConvW c;
  c.cin = cin;
  c.cout = cout;
  c.ks = ks;
  c.cout_pad = round_up(cout, 16);
  c.cout_k = round_up(cout, 64);
  c.cin_rows = round_up(cin, 16);
  const int taps = ks * ks;
  if (cin % 64) throw EngineError(-42, "conv '" + prefix + "': input channels must be a multiple of 64");
  std::vector<float> f((size_t)taps * c.cout_pad * cin, 0.f), d((size_t)taps * c.cin_rows * c.cout_k, 0.f);
  for (int co = 0; co < cout; ++co)
    for (int ci = 0; ci < cin_real; ++ci)
      for (int ty = 0; ty < ks; ++ty)
        for (int tx = 0; tx < ks; ++tx) {
          float v = w.data[(((size_t)co * cin_real + ci) * ks + ty) * ks + tx];
          int t = ty * ks + tx;
          f[((size_t)t * c.cout_pad + co) * cin + ci] = v;
          // dgrad: dx[p] = sum_t dy[p + off(t)] * W[.., flipped t]
          int tf = (ks - 1 - ty) * ks + (ks - 1 - tx);
          d[((size_t)tf * c.cin_rows + ci) * c.cout_k + co] = v;
        }
  c.w = upload_f16(f);
  c.wd = upload_f16(d);
  c.bias = upload(b.data);
  return c;
}

// ===================================================================================================== VQGAN drawer
Engine::GNSaved Engine::add_gn(OpList& l, const Act& x, const NormW& n, int swish, act_t* y) {
  GNSaved s;
  s.stats = dalloc<float>(64);
  s.gstats = dalloc<float>(64);
  const act_t* xp = x.p;
  int px = x.pixels(), C = x.C;
  float* part = gn_part;
  float* stats = s.stats;
  cudaStream_t cs = st;
  NormW nn = n;
  const int nsm = num_sms;
  if (gn_group && gn_group_supported(px, C)) {
    const std::string shape = " px=" + std::to_string(px) + " C=" + std::to_string(C);
    if (const GnSplitK* pk = gn_fuse_fwd ? take_pending_splitk(l, xp, px, C, false) : nullptr) {
      const GnSplitK sk = *pk;
      l.ops.back() = [=] { gn_forward_group(nullptr, &sk, nn.gamma, nn.beta, px, C, swish, 1e-6f, stats, y, cs); };
      l.names.back() = "splitk_reduce+gn_fwd_group" + shape + " splits=" + std::to_string(sk.splits);
      pend_sk.erase(&l);
    } else {
      l.add(1, [=] { gn_forward_group(xp, nullptr, nn.gamma, nn.beta, px, C, swish, 1e-6f, stats, y, cs); }, 0.0,
            "gn_fwd_group" + shape);
    }
  } else if (gn_coop && gn_coop_supported(px, C, nsm)) {
    GridBarrier* gb = &gn_bar;
    l.add(1, [=] { gn_forward_coop(xp, nn.gamma, nn.beta, px, C, swish, 1e-6f, part, stats, y, nsm, gb, cs); }, 0.0,
          "gn_fwd_coop px=" + std::to_string(px) + " C=" + std::to_string(C));
  } else {
    l.add(3, [=] {
      gn_stats(xp, px, C, 1e-6f, part, stats, cs);
      gn_apply(xp, stats, nn.gamma, nn.beta, px, C, swish, y, cs);
    }, 0.0, "gn_fwd_3k px=" + std::to_string(px) + " C=" + std::to_string(C));
  }
  return s;
}

void Engine::add_gn_bwd(OpList& l, const act_t* dy, const act_t* x, const GNSaved& s, const NormW& n, int px, int C,
                        int swish, const act_t* dres, act_t* dx) {
  float* part = gn_part;
  cudaStream_t cs = st;
  const int nsm = num_sms;
  GridBarrier* gb = &gn_bar;
  if (gn_group && gn_group_supported(px, C)) {
    const std::string shape = " px=" + std::to_string(px) + " C=" + std::to_string(C);
    if (const GnSplitK* pk = gn_fuse_bwd ? take_pending_splitk(l, dy, px, C, true) : nullptr) {
      const GnSplitK sk = *pk;  // dy itself is never written: the reduced gradient lives in registers only
      l.ops.back() = [=] { gn_backward_group(nullptr, &sk, x, s.stats, n.gamma, n.beta, px, C, swish, dres, dx, cs); };
      l.names.back() = "splitk_reduce+gn_bwd_group" + shape + " splits=" + std::to_string(sk.splits);
      pend_sk.erase(&l);
    } else {
      l.add(1, [=] { gn_backward_group(dy, nullptr, x, s.stats, n.gamma, n.beta, px, C, swish, dres, dx, cs); }, 0.0,
            "gn_bwd_group" + shape);
    }
  } else if (gn_coop && gn_coop_supported(px, C, nsm))
    l.add(1, [=] { gn_backward_coop(dy, x, s.stats, n.gamma, n.beta, px, C, swish, dres, part, dx, nsm, gb, cs); }, 0.0,
          "gn_bwd_coop px=" + std::to_string(px) + " C=" + std::to_string(C));
  else
    l.add(3, [=] { gn_backward(dy, x, s.stats, n.gamma, n.beta, px, C, swish, dres, part, s.gstats, dx, cs); }, 0.0,
          "gn_bwd_3k px=" + std::to_string(px) + " C=" + std::to_string(C));
}

// y = conv(x) (+bias), returns y; appends dgrad op (x.g = conv_dgrad(y.g)) to bwd (caller orders it)
Act Engine::conv_fwd_bwd(const Act& x, const ConvW& w, OpList& bwd) {
  Act y = new_act(x.H, x.W, w.cout);
  GemmEpilogue e;
  e.bias = w.bias;
  e.out_f16 = y.p;
  e.ldc = y.C;
  add_conv(drawer_fwd, x.p, x.H, x.W, x.C, w.w, w.cout_pad, w.cout, w.ks, e);
  GemmEpilogue d;
  d.out_f16 = x.g;
  d.ldc = x.C;
  add_conv(bwd, y.g, x.H, x.W, w.cout_k, w.wd, w.cin_rows, w.cin, w.ks, d);
  return y;
}

Act Engine::resblock(const Act& x, const std::string& prefix, int cin, int cout) {
  NormW n1 = load_norm(PXR_MOD_VQGAN, prefix + ".norm1", cin), n2 = load_norm(PXR_MOD_VQGAN, prefix + ".norm2", cout);
  ConvW c1 = load_conv(prefix + ".conv1", cin, cout, 3), c2 = load_conv(prefix + ".conv2", cout, cout, 3);
  const int H = x.H, Wd = x.W, px = x.pixels();
  Act a1 = new_act(H, Wd, cin), h1 = new_act(H, Wd, cout), a2 = new_act(H, Wd, cout), out = new_act(H, Wd, cout);
  cudaStream_t cs = st;
  float* part = gn_part;
  // ---- forward
  GNSaved s1 = add_gn(drawer_fwd, x, n1, 1, a1.p);
  {
    GemmEpilogue e;
    e.bias = c1.bias;
    e.out_f16 = h1.p;
    e.ldc = cout;
    add_conv(drawer_fwd, a1.p, H, Wd, cin, c1.w, c1.cout_pad, cout, 3, e);
  }
  GNSaved s2 = add_gn(drawer_fwd, h1, n2, 1, a2.p);
  ConvW sc;
  if (cin != cout) {
    sc = load_conv(prefix + ".nin_shortcut", cin, cout, 1);
    GemmEpilogue e;
    e.bias = sc.bias;
    e.out_f16 = out.p;
    e.ldc = cout;
    add_conv(drawer_fwd, x.p, H, Wd, cin, sc.w, sc.cout_pad, cout, 1, e);
  }
  {
    GemmEpilogue e;
    e.bias = c2.bias;
    e.res_f16 = (cin != cout) ? out.p : x.p;
    e.out_f16 = out.p;
    e.ldc = cout;
    add_conv(drawer_fwd, a2.p, H, Wd, cout, c2.w, c2.cout_pad, cout, 3, e);
  }
  // ---- backward (execution order)
  OpList b;
  {
    GemmEpilogue e;
    e.out_f16 = a2.g;
    e.ldc = cout;
    add_conv(b, out.g, H, Wd, c2.cout_k, c2.wd, c2.cin_rows, cout, 3, e);
  }
  add_gn_bwd(b, a2.g, h1.p, s2, n2, px, cout, 1, nullptr, h1.g);
  {
    GemmEpilogue e;
    e.out_f16 = a1.g;
    e.ldc = cin;
    add_conv(b, h1.g, H, Wd, c1.cout_k, c1.wd, c1.cin_rows, cin, 3, e);
  }
  if (cin != cout) {
    GemmEpilogue e;
    e.out_f16 = x.g;
    e.ldc = cin;
    add_conv(b, out.g, H, Wd, sc.cout_k, sc.wd, sc.cin_rows, cin, 1, e);
    add_gn_bwd(b, a1.g, x.p, s1, n1, px, cin, 1, x.g, x.g);
  } else {
    add_gn_bwd(b, a1.g, x.p, s1, n1, px, cin, 1, out.g, x.g);
  }
  bwd_stack.push_back(std::move(b));
  return out;
}

Act Engine::attnblock(const Act& x, const std::string& prefix, int c) {
  NormW n = load_norm(PXR_MOD_VQGAN, prefix + ".norm", c);
  // fused q/k/v 1x1 convs: weight [3c, c]
  std::vector<float> wq, bq;
  for (const char* nm : {".q", ".k", ".v"}) {
    const HostWeight& w = W(PXR_MOD_VQGAN, prefix + nm + ".weight", {c, c, 1, 1});
    const HostWeight& b = W(PXR_MOD_VQGAN, prefix + nm + ".bias", {c});
    wq.insert(wq.end(), w.data.begin(), w.data.end());
    bq.insert(bq.end(), b.data.begin(), b.data.end());
  }
  act_t* wqkv = upload_f16(wq);
  float* bqkv = upload(bq);
  ConvW po = load_conv(prefix + ".proj_out", c, c, 1);
  const int T = x.pixels(), ldT = round_up(T, 8);
  const float alpha = 1.f / std::sqrt((float)c);
  Act a = new_act(x.H, x.W, c), O = new_act(x.H, x.W, c), out = new_act(x.H, x.W, c);
  act_t* qkv = dalloc<act_t>((size_t)T * 3 * c);
  act_t* gqkv = dalloc<act_t>((size_t)T * 3 * c);
  act_t* P = dalloc<act_t>((size_t)T * ldT);
  act_t* dP = dalloc<act_t>((size_t)T * ldT);
  cudaStream_t cs = st;
  float* part = gn_part;
  // ---- forward
  GNSaved s = add_gn(drawer_fwd, x, n, 0, a.p);
  {
    GemmEpilogue e;
    e.bias = bqkv;
    e.out_f16 = qkv;
    e.ldc = 3 * c;
    add_gemm(drawer_fwd, opK(a.p, c, T, c), opK(wqkv, c, 3 * c, c), T, 3 * c, c, e);
  }
  const bool fuse_sm = fuse_softmax && T <= 256;  // whole row in one accumulator tile -> softmax in the GEMM epilogue
  {
    GemmEpilogue e;
    e.alpha = alpha;
    e.out_f16 = P;
    e.ldc = ldT;
    if (fuse_sm) {
      e.act = ACT_SOFTMAX;
      e.n_store = ldT;
    }
    add_gemm(drawer_fwd, opK(qkv, 3 * c, T, c), opK(qkv + c, 3 * c, T, c), T, T, c, e, fuse_sm ? round_up(T, 16) : 0);
  }
  if (!fuse_sm) drawer_fwd.add(1, [=] { softmax_forward(P, T, T, ldT, cs); }, 0.0, "softmax_forward");
  {
    GemmEpilogue e;
    e.out_f16 = O.p;
    e.ldc = c;
    add_gemm(drawer_fwd, opK(P, ldT, T, ldT), opMN(qkv + 2 * c, 3 * c, c, T), T, c, T, e);
  }
  {
    GemmEpilogue e;
    e.bias = po.bias;
    e.res_f16 = x.p;
    e.out_f16 = out.p;
    e.ldc = c;
    add_conv(drawer_fwd, O.p, x.H, x.W, c, po.w, po.cout_pad, c, 1, e);
  }
  // ---- backward
  OpList b;
  {
    GemmEpilogue e;
    e.out_f16 = O.g;
    e.ldc = c;
    add_conv(b, out.g, x.H, x.W, po.cout_k, po.wd, po.cin_rows, c, 1, e);
  }
  {  // dP = dO v^T ; dS = alpha * P * (dP - <P, dP>) fused in the epilogue when the row fits one tile
    GemmEpilogue e;
    e.out_f16 = dP;
    e.ldc = ldT;
    if (fuse_sm) {
      e.act = ACT_SOFTMAX_BWD;
      e.aux_in = P;
      e.alpha = alpha;
      e.n_store = ldT;
    }
    add_gemm(b, opK(O.g, c, T, c), opK(qkv + 2 * c, 3 * c, T, c), T, T, c, e, fuse_sm ? round_up(T, 16) : 0);
  }
  if (!fuse_sm) b.add(1, [=] { softmax_backward(P, dP, T, T, ldT, cs); }, 0.0, "softmax_backward");
  const float alpha_b = fuse_sm ? 1.f : alpha;  // fused path already carries alpha in dS
  {  // dq = alpha dS k
    GemmEpilogue e;
    e.alpha = alpha_b;
    e.out_f16 = gqkv;
    e.ldc = 3 * c;
    add_gemm(b, opK(dP, ldT, T, ldT), opMN(qkv + c, 3 * c, c, T), T, c, T, e);
  }
  {  // dk = alpha dS^T q
    GemmEpilogue e;
    e.alpha = alpha_b;
    e.out_f16 = gqkv + c;
    e.ldc = 3 * c;
    add_gemm(b, opMN(dP, ldT, T, T), opMN(qkv, 3 * c, c, T), T, c, T, e);
  }
  {  // dv = P^T dO
    GemmEpilogue e;
    e.out_f16 = gqkv + 2 * c;
    e.ldc = 3 * c;
    add_gemm(b, opMN(P, ldT, T, T), opMN(O.g, c, c, T), T, c, T, e);
  }
  {  // da = dqkv Wqkv   (B = Wqkv stored [3c (k), c (n)] -> MN-major)
    GemmEpilogue e;
    e.out_f16 = a.g;
    e.ldc = c;
    add_gemm(b, opK(gqkv, 3 * c, T, 3 * c), opMN(wqkv, c, c, 3 * c), T, c, 3 * c, e);
  }
  add_gn_bwd(b, a.g, x.p, s, n, T, c, 0, out.g, x.g);
  bwd_stack.push_back(std::move(b));
  return out;
}

Act Engine::upsample(const Act& x, const std::string& prefix) {
  ConvW cw = load_conv(prefix + ".conv", x.C, x.C, 3);
  Act u = new_act(2 * x.H, 2 * x.W, x.C);
  cudaStream_t cs = st;
  drawer_fwd.add(1, [=] { upsample2x(x.p, x.H, x.W, x.C, u.p, cs); }, 0.0, "upsample2x");
  OpList b;
  Act out = conv_fwd_bwd(u, cw, b);
  b.add(1, [=] { downsum2x(u.g, x.H, x.W, x.C, x.g, cs); }, 0.0, "downsum2x");
  bwd_stack.push_back(std::move(b));
  return out;
}

void Engine::build_vqgan() {
  const int zc = cfg.z_channels, ne = cfg.n_embed, L = cfg.n_levels;
  if (L < 1 || L > 8) throw EngineError(-43, "n_levels must be in [1, 8]");
  const int f = 1 << (L - 1);
  if (cfg.image_h % f || cfg.image_w % f)
    throw EngineError(-44, "image size must be a multiple of 2^(n_levels-1)");
  const int h = cfg.image_h / f, w = cfg.image_w / f, hw = h * w;
  z_numel = (int64_t)zc * hw;
  // GN scratch sized for the largest activation
  // (the cooperative kernels use up to one block per SM, the three-kernel path gn_num_partials blocks)
  gn_part = dalloc<float>((size_t)std::max(gn_num_partials(cfg.image_h * cfg.image_w, 64), num_sms + 1) * 64 + 64);
  gn_bar.counter = dalloc<unsigned long long>(1);
  splitk_ws_elems = (size_t)8 << 20;  // 32 MiB of fp32 partial sums: covers every conv the split-K rule selects
  splitk_ws = dalloc<float>(splitk_ws_elems, false);
  // codebook
  const HostWeight& cb = W(PXR_MOD_VQGAN, "quantize.embedding.weight", {ne, zc});
  std::vector<float> cbT((size_t)zc * ne), c2(ne), mn(zc, 1e30f), mx(zc, -1e30f);
  for (int j = 0; j < ne; ++j) {
    float s = 0.f;
    for (int k = 0; k < zc; ++k) {
      float v = cb.data[(size_t)j * zc + k];
      cbT[(size_t)k * ne + j] = v;
      s += v * v;  // codebook.pow(2).sum(dim=1), vqgan.py:61
      mn[k] = std::min(mn[k], v);
      mx[k] = std::max(mx[k], v);
    }
    c2[j] = s;
  }
  float* d_cb = upload(cb.data);
  float* d_cbT = upload(cbT);
  float* d_c2 = upload(c2);
  zmin = upload(mn);  // vqgan.py:141-142
  zmax = upload(mx);
  const int n_chunks = (ne + 1023) / 1024;
  float* part_d = dalloc<float>((size_t)hw * n_chunks);
  int* part_i = dalloc<int>((size_t)hw * n_chunks);
  int* idx = dalloc<int>(hw);
  Act zq = new_act(h, w, zc);
  cudaStream_t cs = st;
  float* zb = z_buf = dalloc<float>(z_numel);
  z_grad = dalloc<float>(z_numel);
  bool vq_tc = vq_tc_supported(zc, ne);
  if (const char* e = getenv("PXR_VQ_TC")) vq_tc = vq_tc && atoi(e) != 0;
  if (vq_tc) {
    // distance matrix on the tensor cores, decision in exact fp32 (kernels_vq_tc.cu)
    float amax = 0.f, cmax2 = 0.f, cmax1 = 0.f;
    for (int j = 0; j < ne; ++j) {
      double s2 = 0.0, s1 = 0.0;
      for (int k = 0; k < zc; ++k) {
        const float v = std::fabs(cb.data[(size_t)j * zc + k]);
        amax = std::max(amax, v);
        s2 += (double)v * v;
        s1 += v;
      }
      cmax2 = std::max(cmax2, (float)std::sqrt(s2) * 1.000001f);
      cmax1 = std::max(cmax1, (float)s1 * 1.000001f);
    }
    int ex = 0;
    if (amax > 0.f) std::frexp(amax, &ex);
    const float cb_scale = std::ldexp(1.f, -ex);  // power of two: max |c| lands in [0.5, 1)
    std::vector<float> cbs(cb.data.size());
    for (size_t i = 0; i < cbs.size(); ++i) cbs[i] = cb.data[i] * cb_scale;
    act_t* cbh = upload_f16(cbs);
    act_t* zh = dalloc<act_t>((size_t)hw * zc);
    float* pinfo = dalloc<float>((size_t)hw * 4);
    float* scores = dalloc<float>((size_t)hw * ne, false);
    int* vq_stats = dalloc<int>(2);
    drawer_fwd.add(1, [=] { vq_prep(zb, zc, hw, zh, pinfo, cs); }, 0.0, "vq_prep");
    {
      GemmEpilogue e;
      e.out_f32 = scores;
      e.ldc = ne;
      add_gemm(drawer_fwd, opK(zh, zc, hw, zc), opK(cbh, zc, ne, zc), hw, ne, zc, e);
    }
    drawer_fwd.add(1, [=] { vq_select(scores, ne, zb, d_cb, d_c2, pinfo, cb_scale, cmax2, cmax1, zc, hw, ne, idx, zq.p, vq_stats, cs); },
                   0.0, "vq_select");
    reg("vq_stats", vq_stats, sizeof(int) * 2);  // {candidates rechecked in fp32, positions that fell back to the full search}, cumulative
  } else {
    drawer_fwd.add(2, [=] { vq_nearest(zb, d_cbT, d_c2, d_cb, zc, hw, ne, part_d, part_i, idx, zq.p, cs); }, 0.0, "vq_nearest");
  }
  reg("vq_idx", idx, sizeof(int) * hw);  // argmin code per latent position (vqgan.py:62): integer bookkeeping

  // post_quant_conv + decoder
  ConvW pq = load_conv("post_quant_conv", zc, zc, 1);
  OpList b_in;
  Act hq = conv_fwd_bwd(zq, pq, b_in);
  int block_in = cfg.ch * cfg.ch_mult[L - 1];
  ConvW cin = load_conv("decoder.conv_in", zc, block_in, 3);
  OpList b_in2;
  Act hcur = conv_fwd_bwd(hq, cin, b_in2);
  {
    OpList b;  // execution order: conv_in dgrad, then post_quant dgrad, then vq backward
    b.append(b_in2);
    b.append(b_in);
    float* zg = z_grad;
    float inv = 1.f / S;
    b.add(1, [=] { vq_backward(zq.g, inv, zc, hw, zg, cs); }, 0.0, "vq_backward");
    bwd_stack.push_back(std::move(b));
  }
  hcur = resblock(hcur, "decoder.mid.block_1", block_in, block_in);
  hcur = attnblock(hcur, "decoder.mid.attn_1", block_in);
  hcur = resblock(hcur, "decoder.mid.block_2", block_in, block_in);
  int curr_res = cfg.resolution / f;
  for (int lv = L - 1; lv >= 0; --lv) {
    int block_out = cfg.ch * cfg.ch_mult[lv];
    for (int ib = 0; ib < cfg.num_res_blocks + 1; ++ib) {
      std::string p = "decoder.up." + std::to_string(lv) + ".block." + std::to_string(ib);
      hcur = resblock(hcur, p, block_in, block_out);
      block_in = block_out;
      if (curr_res == cfg.attn_resolution)
        hcur = attnblock(hcur, "decoder.up." + std::to_string(lv) + ".attn." + std::to_string(ib), block_in);
    }
    if (lv != 0) {
      hcur = upsample(hcur, "decoder.up." + std::to_string(lv) + ".upsample");
      curr_res *= 2;
    }
  }
  // norm_out, swish, conv_out -> image
  NormW no = load_norm(PXR_MOD_VQGAN, "decoder.norm_out", block_in);
  ConvW co = load_conv("decoder.conv_out", block_in, 3, 3);
  Act a = new_act(hcur.H, hcur.W, block_in);
  GNSaved s = add_gn(drawer_fwd, hcur, no, 1, a.p);
  const int px = hcur.pixels();
  float* co_out = dalloc<float>((size_t)px * co.cout_pad);
  act_t* co_g = dalloc<act_t>((size_t)px * co.cout_k);
  {
    GemmEpilogue e;
    e.bias = co.bias;
    e.out_f32 = co_out;
    e.ldc = co.cout_pad;
    add_conv(drawer_fwd, a.p, hcur.H, hcur.W, block_in, co.w, co.cout_pad, 3, 3, e);
  }
  img = dalloc<float>((size_t)3 * px);
  img_pre = dalloc<float>((size_t)3 * px);
  g_img = dalloc<float>((size_t)3 * px);
  {
    float *ip = img_pre, *im = img;
    int ld = co.cout_pad;
    drawer_fwd.add(1, [=] { image_finish(co_out, ld, px, ip, im, cs); }, 0.0, "image_finish");
  }
  {
    OpList b;
    float *gi = g_img, *ip = img_pre;
    int ldk = co.cout_k;
    float* part = gn_part;
    b.add(1, [=] { image_finish_backward(gi, ip, px, ldk, co_g, cs); }, 0.0, "image_finish_backward");
    GemmEpilogue e;
    e.out_f16 = a.g;
    e.ldc = block_in;
    add_conv(b, co_g, hcur.H, hcur.W, co.cout_k, co.wd, co.cin_rows, block_in, 3, e);
    Act hc = hcur;
    add_gn_bwd(b, a.g, hc.p, s, no, px, hc.C, 1, nullptr, hc.g);
    bwd_stack.push_back(std::move(b));
  }
  // flatten backward stack in reverse block order
  for (int i = (int)bwd_stack.size() - 1; i >= 0; --i) drawer_bwd.append(bwd_stack[i]);
  bwd_stack.clear();
  if (weights[PXR_MOD_VQGAN].count("encoder.conv_in.weight")) build_vqgan_encoder();
}

// taming Encoder (un-vendored: taming/modules/diffusionmodules/model.py, restated in oracle/ref_path.py): conv_in, per level
// num_res_blocks x ResnetBlock (+ AttnBlock at attn_resolution) and a strided Downsample, mid block_1 / attn_1 / block_2,
// norm_out + swish + conv_out; then VQModel.encode's quant_conv and the quantiser's nearest code.  Same kernels as the
// decoder's forward; no backward (the encoder only runs at init / overlay time, never inside the gradient path).
void Engine::build_vqgan_encoder() {
  const int zc = cfg.z_channels, ne = cfg.n_embed, L = cfg.n_levels, H = cfg.image_h, Wd = cfg.image_w;
  cudaStream_t cs = st;
  auto act = [&](int h, int w, int c) {
    Act a;
    a.H = h;
    a.W = w;
    a.C = c;
    a.p = dalloc<act_t>((size_t)h * w * c);
    return a;
  };
  auto conv = [&](const Act& x, const ConvW& w, const act_t* res) {
    Act y = act(x.H, x.W, w.cout);
    GemmEpilogue e;
    e.bias = w.bias;
    e.res_f16 = res;
    e.out_f16 = y.p;
    e.ldc = y.C;
    add_conv(enc_fwd, x.p, x.H, x.W, x.C, w.w, w.cout_pad, w.cout, w.ks, e);
    return y;
  };
  auto resblock_fwd = [&](const Act& x, const std::string& prefix, int cin, int cout) {
    NormW n1 = load_norm(PXR_MOD_VQGAN, prefix + ".norm1", cin), n2 = load_norm(PXR_MOD_VQGAN, prefix + ".norm2", cout);
    ConvW c1 = load_conv(prefix + ".conv1", cin, cout, 3), c2 = load_conv(prefix + ".conv2", cout, cout, 3);
    Act a1 = act(x.H, x.W, cin), a2 = act(x.H, x.W, cout);
    add_gn(enc_fwd, x, n1, 1, a1.p);
    Act h1 = conv(a1, c1, nullptr);
    add_gn(enc_fwd, h1, n2, 1, a2.p);
    const act_t* shortcut = x.p;
    if (cin != cout) {
      ConvW sc = load_conv(prefix + ".nin_shortcut", cin, cout, 1);
      shortcut = conv(x, sc, nullptr).p;
    }
    return conv(a2, c2, shortcut);
  };
  auto attn_fwd = [&](const Act& x, const std::string& prefix, int c) {
    NormW n = load_norm(PXR_MOD_VQGAN, prefix + ".norm", c);
    std::vector<float> wq, bq;
    for (const char* nm : {".q", ".k", ".v"}) {
      const HostWeight& w = W(PXR_MOD_VQGAN, prefix + nm + ".weight", {c, c, 1, 1});
      const HostWeight& b = W(PXR_MOD_VQGAN, prefix + nm + ".bias", {c});
      wq.insert(wq.end(), w.data.begin(), w.data.end());
      bq.insert(bq.end(), b.data.begin(), b.data.end());
    }
    act_t* wqkv = upload_f16(wq);
    float* bqkv = upload(bq);
    ConvW po = load_conv(prefix + ".proj_out", c, c, 1);
    const int T = x.pixels(), ldT = round_up(T, 8);
    Act a = act(x.H, x.W, c), O = act(x.H, x.W, c);
    act_t* qkv = dalloc<act_t>((size_t)T * 3 * c);
    act_t* P = dalloc<act_t>((size_t)T * ldT);
    add_gn(enc_fwd, x, n, 0, a.p);
    {
      GemmEpilogue e;
      e.bias = bqkv;
      e.out_f16 = qkv;
      e.ldc = 3 * c;
      add_gemm(enc_fwd, opK(a.p, c, T, c), opK(wqkv, c, 3 * c, c), T, 3 * c, c, e);
    }
    {
      GemmEpilogue e;
      e.alpha = 1.f / std::sqrt((float)c);
      e.out_f16 = P;
      e.ldc = ldT;
      add_gemm(enc_fwd, opK(qkv, 3 * c, T, c), opK(qkv + c, 3 * c, T, c), T, T, c, e);
    }
    enc_fwd.add(1, [=] { softmax_forward(P, T, T, ldT, cs); }, 0.0, "softmax_forward");
    {
      GemmEpilogue e;
      e.out_f16 = O.p;
      e.ldc = c;
      add_gemm(enc_fwd, opK(P, ldT, T, ldT), opMN(qkv + 2 * c, 3 * c, c, T), T, c, T, e);
    }
    return conv(O, po, x.p);
  };
  enc_img = dalloc<float>((size_t)3 * H * Wd);
  Act x0 = act(H, Wd, 64);
  {
    float* im = enc_img;
    const int px = H * Wd;
    enc_fwd.add(1, [=] { image_to_nhwc64(im, px, x0.p, cs); }, 0.0, "image_to_nhwc64");
  }
  ConvW cin_w = load_conv("encoder.conv_in", 64, cfg.ch, 3, 3);
  Act hcur = conv(x0, cin_w, nullptr);
  int curr_res = cfg.resolution, block_in = cfg.ch;
  for (int lv = 0; lv < L; ++lv) {
    const int block_out = cfg.ch * cfg.ch_mult[lv];
    for (int ib = 0; ib < cfg.num_res_blocks; ++ib) {
      const std::string p = "encoder.down." + std::to_string(lv) + ".block." + std::to_string(ib);
      hcur = resblock_fwd(hcur, p, block_in, block_out);
      block_in = block_out;
      if (curr_res == cfg.attn_resolution)
        hcur = attn_fwd(hcur, "encoder.down." + std::to_string(lv) + ".attn." + std::to_string(ib), block_in);
    }
    if (lv != L - 1) {
      ConvW dw = load_conv("encoder.down." + std::to_string(lv) + ".downsample.conv", block_in, block_in, 3);
      Act full = conv(hcur, dw, nullptr);
      Act half = act(hcur.H / 2, hcur.W / 2, block_in);
      const int fh = hcur.H, fw = hcur.W, fc = block_in;
      enc_fwd.add(1, [=] { subsample_odd(full.p, fh, fw, fc, half.p, cs); }, 0.0, "subsample_odd");
      hcur = half;
      curr_res /= 2;
    }
  }
  hcur = resblock_fwd(hcur, "encoder.mid.block_1", block_in, block_in);
  hcur = attn_fwd(hcur, "encoder.mid.attn_1", block_in);
  hcur = resblock_fwd(hcur, "encoder.mid.block_2", block_in, block_in);
  NormW no = load_norm(PXR_MOD_VQGAN, "encoder.norm_out", block_in);
  Act a = act(hcur.H, hcur.W, block_in);
  add_gn(enc_fwd, hcur, no, 1, a.p);
  ConvW co = load_conv("encoder.conv_out", block_in, zc, 3);  // double_z = False for the VQ models
  Act hz = conv(a, co, nullptr);
  ConvW qc = load_conv("quant_conv", zc, zc, 1);
  Act hq = conv(hz, qc, nullptr);
  const int hw = hq.pixels();
  if ((int64_t)zc * hw != z_numel) throw EngineError(-44, "encoder output does not match the latent size");
  // quantise: the same exact fp32 nearest-code search as synth (the codebook copies are the decoder's)
  const HostWeight& cb = W(PXR_MOD_VQGAN, "quantize.embedding.weight", {ne, zc});
  std::vector<float> cbT((size_t)zc * ne), c2(ne);
  for (int j = 0; j < ne; ++j) {
    float s2 = 0.f;
    for (int k = 0; k < zc; ++k) {
      const float v = cb.data[(size_t)j * zc + k];
      cbT[(size_t)k * ne + j] = v;
      s2 += v * v;
    }
    c2[j] = s2;
  }
  float *d_cb = upload(cb.data), *d_cbT = upload(cbT), *d_c2 = upload(c2);
  const int n_chunks = (ne + 1023) / 1024;
  float* part_d = dalloc<float>((size_t)hw * n_chunks);
  int* part_i = dalloc<int>((size_t)hw * n_chunks);
  int* idx = dalloc<int>(hw);
  float* z32 = dalloc<float>((size_t)zc * hw);
  act_t* zq16 = dalloc<act_t>((size_t)hw * zc);
  enc_z = dalloc<float>((size_t)zc * hw);
  float* ez = enc_z;
  enc_fwd.add(4, [=] {
    vq_backward(hq.p, 1.f, zc, hw, z32, cs);  // NHWC fp16 -> [C, hw] fp32 (the same transpose kernel the decoder's backward ends with)
    vq_nearest(z32, d_cbT, d_c2, d_cb, zc, hw, ne, part_d, part_i, idx, zq16, cs);
    gather_codes(d_cb, idx, zc, hw, ez, cs);
  }, 0.0, "encoder quantise");
  reg("enc_idx", idx, sizeof(int) * hw);
  reg("enc_h", z32, sizeof(float) * zc * hw);
  have_encoder = true;
}

void Engine::build_pixel() {
  const int rows = cfg.grid_rows, cols = cfg.grid_cols, H = cfg.image_h, Wd = cfg.image_w;
  if (rows < 1 || cols < 1) throw EngineError(-46, "pixel drawer needs grid_rows / grid_cols");
  z_numel = (int64_t)3 * rows * cols;
  z_buf = dalloc<float>(z_numel);
  z_grad = dalloc<float>(z_numel);
  img = dalloc<float>((size_t)3 * H * Wd);
  img_pre = dalloc<float>((size_t)3 * H * Wd);
  g_img = dalloc<float>((size_t)3 * H * Wd);
  cudaStream_t cs = st;
  float *zb = z_buf, *ip = img_pre, *im = img, *gi = g_img, *zg = z_grad;
  float inv = 1.f / S;
  drawer_fwd.add(1, [=] { pixel_synth(zb, rows, cols, H, Wd, ip, im, cs); }, 0.0, "pixel_synth");
  drawer_bwd.add(1, [=] { pixel_synth_backward(gi, ip, rows, cols, H, Wd, inv, zg, cs); }, 0.0, "pixel_synth_backward");
}

// FftDrawer.synth (fftdrawer.py:78-84): params = rfft2 spectrum [1,3,H,W/2+1,2]; see kernels_fft.cu
void Engine::build_fft() {
  const int H = cfg.image_h, Wd = cfg.image_w, W2 = Wd / 2 + 1;
  if (Wd % 2) throw EngineError(-48, "fft drawer needs an even canvas width");
  const float decay = cfg.fft_decay > 0 ? cfg.fft_decay : 1.5f, colors = cfg.fft_colors > 0 ? cfg.fft_colors : 1.5f;
  const float contrast = cfg.fft_contrast > 0 ? cfg.fft_contrast : 0.9f;
  const char* msg = nullptr;
  fft = fft_plans_create(H, Wd, st, &msg);
  if (!fft) throw EngineError(-49, msg ? msg : "cuFFT unavailable");
  z_numel = (int64_t)3 * H * W2 * 2;
  // aphantasia fft_image: scale = 1 / max(|f|, 4 / max(h, w)) ** decay * sqrt(w * h) on the rfft2 frequency grid
  std::vector<float> sc((size_t)H * W2);
  for (int y = 0; y < H; ++y) {
    const double fy = (y < (H + 1) / 2 ? y : y - H) / (double)H;  // np.fft.fftfreq
    for (int x = 0; x < W2; ++x) {
      const double fx = (x < (Wd + 1) / 2 ? x : x - Wd) / (double)Wd;
      const double f = std::sqrt(fx * fx + fy * fy);
      sc[(size_t)y * W2 + x] = (float)(1.0 / std::pow(std::max(f, 4.0 / std::max(H, Wd)), (double)decay) * std::sqrt((double)Wd * H));
    }
  }
  // to_valid_rgb: colour-correlation matrix, first column / colors, normalised by the largest column norm
  const double base[3][3] = {{0.26, 0.09, 0.02}, {0.27, 0.00, -0.05}, {0.27, -0.09, 0.03}};
  double m[3][3], maxn = 0;
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 3; ++c) m[r][c] = base[r][c] / (c == 0 ? colors : 1.0);
  for (int c = 0; c < 3; ++c) maxn = std::max(maxn, std::sqrt(m[0][c] * m[0][c] + m[1][c] * m[1][c] + m[2][c] * m[2][c]));
  std::vector<float> M(9);
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 3; ++c) M[r * 3 + c] = (float)(m[r][c] / maxn);
  float* d_scale = upload(sc);
  float* d_M = upload(M);
  const size_t px = (size_t)H * Wd;
  z_buf = dalloc<float>(z_numel);
  z_grad = dalloc<float>(z_numel);
  img = dalloc<float>(3 * px);
  img_pre = dalloc<float>(3 * px);  // irfft output x (unnormalised)
  g_img = dalloc<float>(3 * px);
  float* scaled = dalloc<float>(z_numel);
  float* g1 = dalloc<float>(3 * px);
  float* G = dalloc<float>(z_numel);
  double* part = dalloc<double>(2 * 296 + 8);
  float* stats = dalloc<float>(4);
  cudaStream_t cs = st;
  FftPlans* pl = fft;
  float *zb = z_buf, *x = img_pre, *im = img, *gi = g_img, *zg = z_grad;
  const float inv = 1.f / S;
  drawer_fwd.add(5, [=] { fft_synth_forward(pl, zb, d_scale, d_M, contrast, scaled, x, part, stats, im, cs); }, 0.0, "fft_synth_forward");
  drawer_bwd.add(4, [=] { fft_synth_backward(pl, gi, im, x, d_scale, d_M, contrast, stats, g1, G, part, inv, zg, cs); }, 0.0, "fft_synth_backward");
}

// ===================================================================================================== cutouts
void Engine::build_cutouts() {
  const int cs_ = cfg.cut_size;
  pooled = dalloc<float>((size_t)3 * cs_ * cs_);
  g_pooled = dalloc<float>((size_t)3 * cs_ * cs_);
  pooled_masked = dalloc<float>((size_t)3 * cs_ * cs_);
  aspect = (cfg.cut_aspect > 0.f && cfg.cut_aspect != 1.f) ? (double)cfg.cut_aspect : 1.0;
  if (aspect > 8.0 || aspect < 0.125) throw EngineError(-66, "cut_aspect (canvas width / height) must be within [1/8, 8]");
  source_size(cs_, aspect, src_h, src_w);
  if (aspect != 1.0 && cfg.cut_src_h > 0 && cfg.cut_src_w > 0) {  // the caller's (double-precision) truncation wins
    if (std::abs(cfg.cut_src_h - src_h) > 1 || std::abs(cfg.cut_src_w - src_w) > 1)
      throw EngineError(-66, "cut_src_h / cut_src_w do not match cut_aspect");
    src_h = cfg.cut_src_h;
    src_w = cfg.cut_src_w;
  }
  if (aspect != 1.0) {
    cut_src = dalloc<float>((size_t)3 * src_h * src_w);
    g_cut_src = dalloc<float>((size_t)3 * src_h * src_w);
  } else {
    cut_src = pooled;
    g_cut_src = g_pooled;
  }
  grad_fx = dalloc<long long>((size_t)3 * std::max(src_h * src_w, cs_ * cs_));  // zeroed; each use clears it again
  pool_argmax = dalloc<int>((size_t)3 * cs_ * cs_);
  batch = dalloc<float>((size_t)n_local * 3 * cs_ * cs_);
  g_batch = dalloc<float>((size_t)n_local * 3 * cs_ * cs_);
  n_parts = cutout_num_blocks(n_local, cs_);
  part_min = dalloc<float>(n_parts);
  part_max = dalloc<float>(n_parts);
  part_imin = dalloc<int>(n_parts);
  part_imax = dalloc<int>(n_parts);
  range = dalloc<float>(4);
  irange = dalloc<int>(4);
  sums = dalloc<float>(4);
  sums_fx = dalloc<long long>(2);  // zero-initialised; every pass leaves it zeroed again
  fx_poison = dalloc<unsigned int>(2);
  xbuf = dalloc<float>(4);
  minv_dev = dalloc<float>((size_t)n_local * 12);  // 9 homography + 3 ColorJitter floats per cutout, one H2D copy
  facs_dev = dalloc<float>(n_local);
  for (int i = 0; i < RING; ++i) {
    PXR_CUDA(cudaMallocHost((void**)&minv_host[i], sizeof(float) * n_local * 12));
    PXR_CUDA(cudaMallocHost((void**)&facs_host[i], sizeof(float) * n_local));
    PXR_CUDA(cudaEventCreateWithFlags(&ring_ev[i], cudaEventDisableTiming));
  }
  memset(&cut_args, 0, sizeof cut_args);
  cut_args.pooled = cut_src;
  cut_args.src_h = src_h;
  cut_args.src_w = src_w;
  cut_args.minv = minv_dev;
  cut_args.cs = cs_;
  cut_args.n_local = n_local;
  cut_args.first_global = first_global;
  cut_args.cutn_zoom = (int)(0.6 * cfg.cutn);  // pixray.py:407
  cut_args.seed = cfg.seed;
  cut_args.noise_fac = cfg.noise_fac;
}

// Host side of MakeCutouts: invert the cached "dst <- src" transforms (pixray.py:498) to the sampling maps the
// kernel uses (kornia warp_perspective inverts the normalised homography; with align_corners=True the
// normalisations cancel and src_pix = M^-1 dst_pix), stage them through pinned memory.
void Engine::prepare_cut_params(const pxr_cut_params* p, int iter) {
  // engine-drawn parameters are keyed by (seed, rng_iter): pass b > 0 of an iteration (batches > 1) draws a fresh set,
  // like a second ascend_txt call does, while the padding mode still follows the iteration's parity (pixray.py:1250)
  const int key = rng_iter ? rng_iter : iter;
  const int slot = ring_pos;
  ring_pos = (ring_pos + 1) % RING;
  PXR_CUDA(cudaEventSynchronize(ring_ev[slot]));
  std::vector<float> gen;
  const float* T = p ? p->transforms : nullptr;
  int zoom_padding = p ? p->zoom_padding : ((iter % 2 == 0) ? PXR_PAD_REFLECTION : PXR_PAD_BORDER);  // pixray.py:1250
  float fill = p ? p->fill : 0.f;
  if (!T) {  // engine RNG (SURVEY.md Appendix A), keyed by (seed, iter, global cutout index)
    gen.resize((size_t)cfg.cutn * 9);
    sample_cutout_transforms(cfg.seed, key, cfg.cutn, cfg.cut_size, gen.data(), aspect, src_h, src_w);
    T = gen.data();
    if (!p) fill = sample_fill(cfg.seed, key);
  }
  for (int n = 0; n < n_local; ++n) {
    double m[9], inv[9];
    for (int i = 0; i < 9; ++i) m[i] = T[(size_t)(first_global + n) * 9 + i];
    if (!invert3x3(m, inv)) throw EngineError(-60, "singular cutout transform");
    for (int i = 0; i < 9; ++i) minv_host[slot][n * 9 + i] = (float)inv[i];
  }
  // ColorJitter rows: explicit, or drawn like the transforms when those are the engine's own
  const float* J = p ? p->color_jitter : nullptr;
  std::vector<float> genj;
  if (!J && !(p && p->transforms) && cj_p > 0.f) {
    genj.resize((size_t)cfg.cutn * 3);
    sample_color_jitter(cfg.seed, key, cfg.cutn, cj_p, cj_sat, cj_hue, genj.data());
    J = genj.data();
  }
  float* jh = minv_host[slot] + (size_t)n_local * 9;
  if (J)
    for (int i = 0; i < n_local * 3; ++i) jh[i] = J[(size_t)first_global * 3 + i];
  cut_args.jitter = J ? minv_dev + (size_t)n_local * 9 : nullptr;
  PXR_CUDA(cudaMemcpyAsync(minv_dev, minv_host[slot], sizeof(float) * n_local * (J ? 12 : 9), cudaMemcpyHostToDevice, st));
  cut_args.zoom_padding = zoom_padding;
  cut_args.fill = fill;
  cut_args.iter = key;
  cut_args.noise = nullptr;
  cut_args.noise_facs = nullptr;
  if (cfg.noise_fac <= 0.f) {
    cut_args.noise_mode = 0;
  } else if (p && p->noise && p->noise_facs) {
    for (int n = 0; n < n_local; ++n) facs_host[slot][n] = p->noise_facs[first_global + n];
    PXR_CUDA(cudaMemcpyAsync(facs_dev, facs_host[slot], sizeof(float) * n_local, cudaMemcpyHostToDevice, st));
    cut_args.noise_mode = 1;
    cut_args.noise = p->noise + (size_t)first_global * 3 * cfg.cut_size * cfg.cut_size;
    cut_args.noise_facs = facs_dev;
  } else if (p && (p->noise || p->noise_facs)) {
    throw EngineError(-61, "pxr_cut_params: noise and noise_facs must be given together");
  } else if (p && p->transforms) {
    cut_args.noise_mode = 0;  // explicit transforms without noise: deterministic replay
  } else {
    cut_args.noise_mode = 2;
  }
  PXR_CUDA(cudaEventRecord(ring_ev[slot], st));
}

void Engine::forward_cutouts() {
  if (!aux.empty())  // the cutout / embedding losses accumulate per-rank partial sums into their slots
    PXR_CUDA(cudaMemsetAsync(losses_dev + aux_base(), 0, sizeof(float) * aux.size(), st));
  pool_forward(cur_cut_img(), cur_cut_h(), cur_cut_w(), cfg.cut_size, pooled, pool_argmax, st);
  if (aspect != 1.0) {
    rescale_bilinear(pooled, cfg.cut_size, cfg.cut_size, src_h, src_w, cut_src, st);
    launches += 1;
  }
  cutout_forward(cut_args, batch, part_min, part_max, part_imin, part_imax, st);
  minmax_reduce(nullptr, part_min, part_max, part_imin, part_imax, n_parts, range, irange, st);
  launches += 3;
  if (comm) {  // global min / max over all ranks' cutouts (slip.py:21-36 reduces over the whole batch)
    range_pack(range, xbuf, st);
    nccl_check(Comm::api().all_reduce(xbuf, xbuf, 2, Comm::kFloat32, Comm::kMin, comm, st), "allreduce(min,max)");
    range_unpack(xbuf, range, irange, st);
    launches += 3;
  }
  check_launch("cutouts forward");
}

// ===================================================================================================== CLIP ViT
void Engine::build_clip(int i) {
  Clip& C = clip[i];
  C.c = cfg.clip[i];
  const int mod = PXR_MOD_CLIP0 + i;
  const int Wd = C.c.width, L = C.c.layers, Hh = C.c.heads, P = C.c.patch, D = C.c.out_dim;
  if (C.c.image_res != cfg.cut_size) throw EngineError(-50, "clip image_res must equal cut_size");
  if (Wd % 64 || Wd > 1024 || Wd / Hh != 64) throw EngineError(-51, "ViT width must be a multiple of 64 (<=1024) with 64-wide heads");
  if (P < 2 || cfg.cut_size % P) throw EngineError(-52, "patch size must divide cut_size");
  const int gp = cfg.cut_size / P, np = gp * gp, T = np + 1, B = n_local, M = B * T, d = 64;
  const int Kp = round_up(3 * P * P, 64), ldT = round_up(T, 8);
  C.T = T;
  C.np = np;
  C.Kp = Kp;
  C.ldT = ldT;
  C.M = M;
  C.B = B;
  cudaStream_t cs = st;
  // ---- weights
  {
    const HostWeight& w = W(mod, "visual.conv1.weight", {Wd, 3, P, P});
    std::vector<float> f((size_t)Wd * Kp, 0.f);
    for (int o = 0; o < Wd; ++o)
      for (int k = 0; k < 3 * P * P; ++k) f[(size_t)o * Kp + k] = w.data[(size_t)o * 3 * P * P + k];
    C.conv1 = upload_f16(f);
  }
  C.cls = upload(W(mod, "visual.class_embedding", {Wd}).data);
  C.pos = upload(W(mod, "visual.positional_embedding", {T, Wd}).data);
  C.proj = upload(W(mod, "visual.proj", {Wd, D}).data);
  C.proj16 = upload_f16(W(mod, "visual.proj", {Wd, D}).data);
  C.ln_pre = load_norm(mod, "visual.ln_pre", Wd);
  C.ln_post = load_norm(mod, "visual.ln_post", Wd);
  // ---- buffers
  C.patches = dalloc<act_t>((size_t)B * np * Kp);
  C.g_patches = dalloc<act_t>((size_t)B * np * Kp);
  C.t = dalloc<float>((size_t)M * Wd);
  {  // class-token rows are constant: t[b*T + 0] = class_embedding
    std::vector<float> t0((size_t)M * Wd, 0.f);
    const auto& cls = W(mod, "visual.class_embedding").data;
    for (int b = 0; b < B; ++b)
      for (int k = 0; k < Wd; ++k) t0[(size_t)b * T * Wd + k] = cls[k];
    PXR_CUDA(cudaMemcpyAsync(C.t, t0.data(), t0.size() * sizeof(float), cudaMemcpyHostToDevice, st));
    PXR_CUDA(cudaStreamSynchronize(st));
  }
  C.h16 = dalloc<act_t>((size_t)M * Wd);
  C.o16 = dalloc<act_t>((size_t)M * Wd);
  C.gact = dalloc<act_t>((size_t)M * 4 * Wd);
  C.g4 = dalloc<act_t>((size_t)M * 4 * Wd);
  C.gh = dalloc<act_t>((size_t)M * Wd);
  C.go = dalloc<act_t>((size_t)M * Wd);
  C.gqkv = dalloc<act_t>((size_t)M * 3 * Wd);
  const bool fuse_attn = fused_attn && attn_supported(T, d, Wd);  // attn_tc.cu: one kernel per direction, T <= 256
  C.dP = fuse_attn ? nullptr : dalloc<act_t>((size_t)B * Hh * T * ldT);
  const bool s16 = stream16;
  const size_t xbytes = (size_t)M * Wd * (s16 ? sizeof(act_t) : sizeof(float));
  auto xalloc = [&]() -> void* { return dalloc<unsigned char>(xbytes); };
  // fp16 stream: its gradient lives in gx16 alone; fp32 stream: fp32 master gx + the fp16 copy the dgrad GEMMs read
  C.gx = s16 ? nullptr : dalloc<float>((size_t)M * Wd);
  C.gx16 = dalloc<act_t>((size_t)M * Wd);
  C.stats_pre = dalloc<float>((size_t)M * 2);
  C.stats_post = dalloc<float>((size_t)B * 2);
  C.e = dalloc<float>((size_t)B * D);
  C.e_unit = dalloc<float>((size_t)B * D);
  C.de = dalloc<float>((size_t)B * D);
  C.de16 = dalloc<act_t>((size_t)B * D);
  C.hcls = dalloc<act_t>((size_t)B * Wd);
  C.gcls = dalloc<act_t>((size_t)B * Wd);
  void* x_cur = xalloc();
  void* x0 = x_cur;
  // LayerNorm on either stream type
  auto ln_fwd = [s16, cs](const void* x, long long stride, const float* pos, int T_, const NormW& nw, int rows, int W_,
                          act_t* y16, float* y32, float* stats) {
    if (s16) layernorm_forward(static_cast<const act_t*>(x), stride, pos, T_, nw.gamma, nw.beta, rows, W_, 1e-5f, y16, y32, stats, cs);
    else layernorm_forward(static_cast<const float*>(x), stride, pos, T_, nw.gamma, nw.beta, rows, W_, 1e-5f, y16, y32, stats, cs);
  };
  auto ln_bwd = [s16, cs](const act_t* dy, const void* x, long long stride, const float* stats, const NormW& nw, int rows,
                          int W_, int accumulate, float* gx, act_t* gx16) {
    if (s16) layernorm_backward(dy, static_cast<const act_t*>(x), stride, nullptr, 1, stats, nw.gamma, rows, W_, accumulate, gx, gx16, cs);
    else layernorm_backward(dy, static_cast<const float*>(x), stride, nullptr, 1, stats, nw.gamma, rows, W_, accumulate, gx, gx16, cs);
  };
  // residual epilogue x_out = x_res + A B^T + bias on either stream type
  auto residual_epilogue = [s16](GemmEpilogue& e, const void* res, void* out) {
    if (s16) {
      e.res_f16 = static_cast<const act_t*>(res);
      e.out_f16 = static_cast<act_t*>(out);
    } else {
      e.res_f32 = static_cast<const float*>(res);
      e.out_f32 = static_cast<float*>(out);
    }
  };
  C.layers.resize(L);
  const float scale = 1.f / std::sqrt((float)d);
  const bool fuse_sm = fuse_softmax && T <= 256;  // attention row fits one tile: softmax fused into the GEMM epilogue
  const int bnS = fuse_sm ? round_up(T, 16) : pick_bn(T, false, 1000);

  // ---- forward: patch embed (conv1 as GEMM over im2col'd patches, written straight into the token rows 1..np)
  {
    GemmEpilogue e;
    e.out_f32 = C.t + Wd;
    e.ldc = Wd;
    e.bs0 = (long long)T * Wd;
    add_gemm(C.fwd, opK(C.patches, Kp, np, Kp, B, (long long)np * Kp), opK(C.conv1, Kp, Wd, Kp), np, Wd, Kp, e);
  }
  {
    Clip* c = &C;
    void* xo = x0;
    C.fwd.add(1, [=] {
      layernorm_forward(c->t, Wd, c->pos, T, c->ln_pre.gamma, c->ln_pre.beta, M, Wd, 1e-5f, s16 ? static_cast<act_t*>(xo) : nullptr,
                        s16 ? nullptr : static_cast<float*>(xo), c->stats_pre, cs);
    }, 0.0, "layernorm_forward");
  }
  for (int l = 0; l < L; ++l) {
    Clip::Layer& Ly = C.layers[l];
    std::string p = "visual.transformer.resblocks." + std::to_string(l);
    Ly.wqkv = upload_f16(W(mod, p + ".attn.in_proj_weight", {3 * Wd, Wd}).data);
    Ly.bqkv = upload(W(mod, p + ".attn.in_proj_bias", {3 * Wd}).data);
    Ly.wo = upload_f16(W(mod, p + ".attn.out_proj.weight", {Wd, Wd}).data);
    Ly.bo = upload(W(mod, p + ".attn.out_proj.bias", {Wd}).data);
    Ly.wfc = upload_f16(W(mod, p + ".mlp.c_fc.weight", {4 * Wd, Wd}).data);
    Ly.bfc = upload(W(mod, p + ".mlp.c_fc.bias", {4 * Wd}).data);
    Ly.wproj = upload_f16(W(mod, p + ".mlp.c_proj.weight", {Wd, 4 * Wd}).data);
    Ly.bproj = upload(W(mod, p + ".mlp.c_proj.bias", {Wd}).data);
    Ly.ln1 = load_norm(mod, p + ".ln_1", Wd);
    Ly.ln2 = load_norm(mod, p + ".ln_2", Wd);
    Ly.x_in = x_cur;
    Ly.x_mid = xalloc();
    void* x_next = xalloc();
    Ly.stats1 = dalloc<float>((size_t)M * 2);
    Ly.stats2 = dalloc<float>((size_t)M * 2);
    Ly.qkv = dalloc<act_t>((size_t)M * 3 * Wd);
    Ly.P = fuse_attn ? nullptr : dalloc<act_t>((size_t)B * Hh * T * ldT);
    Ly.u = dalloc<act_t>((size_t)M * 4 * Wd);
    if (fuse_attn) {
      Ly.o = dalloc<act_t>((size_t)M * Wd);
      Ly.lse = dalloc<float>((size_t)B * Hh * T);
      Ly.attn = std::make_shared<AttnPlan>();
      char buf[256] = {0};
      int rc = attn_plan_make(Ly.attn.get(), Ly.qkv, Ly.o, C.go, C.gqkv, Ly.lse, B, T, Hh, Wd, scale, num_sms, buf,
                              sizeof buf);
      if (rc) throw EngineError(rc, std::string("attention plan: ") + buf);
    }
    Clip::Layer ly = Ly;
    Clip* c = &C;
    C.fwd.add(1, [=] { ln_fwd(ly.x_in, Wd, nullptr, T, ly.ln1, M, Wd, c->h16, nullptr, ly.stats1); }, 0.0, "layernorm_forward");
    {
      GemmEpilogue e;
      e.bias = ly.bqkv;
      e.out_f16 = ly.qkv;
      e.ldc = 3 * Wd;
      add_gemm(C.fwd, opK(C.h16, Wd, M, Wd), opK(ly.wqkv, Wd, 3 * Wd, Wd), M, 3 * Wd, Wd, e);
    }
    const long long qs0 = d, qs1 = (long long)T * 3 * Wd;           // (head, image) strides inside qkv
    const long long ps0 = (long long)T * ldT, ps1 = (long long)Hh * T * ldT;  // inside P / dP
    const long long os0 = d, os1 = (long long)T * Wd;              // inside [M, W] token-major buffers
    if (fuse_attn) {  // S, softmax and PV in one kernel; S / P never leave the SM
      std::shared_ptr<AttnPlan> ap = ly.attn;
      char lab[96];
      snprintf(lab, sizeof lab, "attn_fwd B=%d T=%d heads=%d", B, T, Hh);
      C.fwd.add(1, [ap, cs] { attn_forward_launch(*ap, cs); }, ap->flops_fwd, lab, ap->bytes_fwd);
    } else {
    {  // S = scale * q k^T  (nn.MultiheadAttention scales q by d^-1/2)
      GemmEpilogue e;
      e.alpha = scale;
      e.out_f16 = ly.P;
      e.ldc = ldT;
      e.bs0 = ps0;
      e.bs1 = ps1;
      if (fuse_sm) {
        e.act = ACT_SOFTMAX;
        e.n_store = ldT;
      }
      add_gemm(C.fwd, opK(ly.qkv, 3 * Wd, T, d, Hh, qs0, B, qs1), opK(ly.qkv + Wd, 3 * Wd, T, d, Hh, qs0, B, qs1), T, T,
               d, e, bnS);
    }
    if (!fuse_sm) C.fwd.add(1, [=] { softmax_forward(ly.P, B * Hh * T, T, ldT, cs); }, 0.0, "softmax_forward");
    {  // O = P v
      GemmEpilogue e;
      e.out_f16 = C.o16;
      e.ldc = Wd;
      e.bs0 = os0;
      e.bs1 = os1;
      add_gemm(C.fwd, opK(ly.P, ldT, T, ldT, Hh, ps0, B, ps1), opMN(ly.qkv + 2 * Wd, 3 * Wd, d, T, Hh, qs0, B, qs1), T, d,
               T, e, 64);
    }
    }
    // Last layer: only the class token's row of every image reaches ln_post / proj (slip.py:62-66 ->
    // VisionTransformer.forward takes x[:, 0, :]), and everything after the attention is row-wise -- out_proj, ln_2, the MLP
    // and their backward run on those B rows (row pitch T * W inside the [M, W] buffers) instead of on all M = B T rows.
    // Exact: the other rows' outputs are never read and their gradients are zero.  PXR_CLIP_LAST_CLS=0 computes all rows.
    const bool cls_only = clip_last_cls && l == L - 1;
    const int Mr = cls_only ? B : M;                                     // rows of the row-wise tail of this layer
    const long long xld = cls_only ? (long long)T * Wd : (long long)Wd;   // their pitch inside the token-major buffers
    {  // x_mid = x_in + O Wo^T + bo
      GemmEpilogue e;
      e.bias = ly.bo;
      residual_epilogue(e, ly.x_in, ly.x_mid);
      e.ldc = xld;
      add_gemm(C.fwd, opK(fuse_attn ? ly.o : C.o16, xld, Mr, Wd), opK(ly.wo, Wd, Wd, Wd), Mr, Wd, Wd, e);
    }
    C.fwd.add(1, [=] { ln_fwd(ly.x_mid, xld, nullptr, T, ly.ln2, Mr, Wd, c->h16, nullptr, ly.stats2); }, 0.0, "layernorm_forward");
    {  // gact = quickgelu(h Wfc^T + bfc), keep pre-activation u   (h16 / gact / u hold the Mr rows compactly)
      GemmEpilogue e;
      e.bias = ly.bfc;
      e.act = ACT_QUICKGELU;
      e.aux_out = ly.u;
      e.out_f16 = C.gact;
      e.ldc = 4 * Wd;
      add_gemm(C.fwd, opK(C.h16, Wd, Mr, Wd), opK(ly.wfc, Wd, 4 * Wd, Wd), Mr, 4 * Wd, Wd, e);
    }
    {  // x_next = x_mid + gact Wproj^T + bproj
      GemmEpilogue e;
      e.bias = ly.bproj;
      residual_epilogue(e, ly.x_mid, x_next);
      e.ldc = xld;
      add_gemm(C.fwd, opK(C.gact, 4 * Wd, Mr, 4 * Wd), opK(ly.wproj, 4 * Wd, Wd, 4 * Wd), Mr, Wd, 4 * Wd, e);
    }
    x_cur = x_next;
  }
  C.x_out = x_cur;
  {  // head: ln_post on the class-token rows (row stride T*W), then e = ln @ proj as a GEMM (proj [W, D] is MN-major)
    Clip* c = &C;
    C.fwd.add(1, [=] { ln_fwd(c->x_out, (long long)T * Wd, nullptr, T, c->ln_post, B, Wd, c->hcls, nullptr, c->stats_post); }, 0.0, "layernorm_forward");
    GemmEpilogue e;
    e.out_f32 = C.e;
    e.ldc = D;
    add_gemm(C.fwd, opK(C.hcls, Wd, B, Wd), opMN(C.proj16, D, D, Wd), B, D, Wd, e);
  }

  // ---- backward (execution order).  Weight operands of the dgrad GEMMs are MN-major views of the forward weights.
  {  // head backward: gcls = de proj^T (proj [W, D] read K-major: n = W rows, k = D), then LN backward on class rows
    Clip* c = &C;
    GemmEpilogue e;
    e.out_f16 = C.gcls;
    e.ldc = Wd;
    add_gemm(C.bwd, opK(C.de16, D, B, D), opK(C.proj16, D, Wd, D), B, Wd, D, e);
    const size_t nbytes32 = (size_t)M * Wd * sizeof(float), nbytes16 = (size_t)M * Wd * sizeof(act_t);
    C.bwd.add(1, [=] {
      if (c->gx) cudaMemsetAsync(c->gx, 0, nbytes32, cs);
      cudaMemsetAsync(c->gx16, 0, nbytes16, cs);
      ln_bwd(c->gcls, c->x_out, (long long)T * Wd, c->stats_post, c->ln_post, B, Wd, 0, c->gx, c->gx16);
    });
  }
  for (int l = L - 1; l >= 0; --l) {
    Clip::Layer ly = C.layers[l];
    Clip* c = &C;
    const long long qs0 = d, qs1 = (long long)T * 3 * Wd, ps0 = (long long)T * ldT, ps1 = (long long)Hh * T * ldT;
    const long long os0 = d, os1 = (long long)T * Wd;
    const bool cls_only = clip_last_cls && l == L - 1;  // see the forward: the row-wise tail of the last layer, class rows only
    const int Mr = cls_only ? B : M;
    const long long xld = cls_only ? (long long)T * Wd : (long long)Wd;
    {  // g4 = (gx Wproj) * quickgelu'(u)
      GemmEpilogue e;
      e.act = ACT_QUICKGELU_BWD;
      e.aux_in = ly.u;
      e.out_f16 = C.g4;
      e.ldc = 4 * Wd;
      add_gemm(C.bwd, opK(C.gx16, xld, Mr, Wd), opMN(ly.wproj, 4 * Wd, 4 * Wd, Wd), Mr, 4 * Wd, Wd, e);
    }
    {  // gh = g4 Wfc
      GemmEpilogue e;
      e.out_f16 = C.gh;
      e.ldc = Wd;
      add_gemm(C.bwd, opK(C.g4, 4 * Wd, Mr, 4 * Wd), opMN(ly.wfc, Wd, Wd, 4 * Wd), Mr, Wd, 4 * Wd, e);
    }
    C.bwd.add(1, [=] { ln_bwd(c->gh, ly.x_mid, xld, ly.stats2, ly.ln2, Mr, Wd, 1, c->gx, c->gx16); }, 0.0, "layernorm_backward");
    if (cls_only) {  // the attention backward reads dO = go for every token: zero outside the class rows
      const size_t go_bytes = (size_t)M * Wd * sizeof(act_t);
      C.bwd.add(1, [=] { cudaMemsetAsync(c->go, 0, go_bytes, cs); }, 0.0, "memset go");
    }
    {  // go = gx Wo
      GemmEpilogue e;
      e.out_f16 = C.go;
      e.ldc = xld;
      add_gemm(C.bwd, opK(C.gx16, xld, Mr, Wd), opMN(ly.wo, Wd, Wd, Wd), Mr, Wd, Wd, e);
    }
    if (fuse_attn) {  // dQ, dK, dV in one kernel (recomputes P from Q, K and the saved log-sum-exp)
      std::shared_ptr<AttnPlan> ap = ly.attn;
      char lab[96];
      snprintf(lab, sizeof lab, "attn_bwd B=%d T=%d heads=%d", B, T, Hh);
      C.bwd.add(1, [ap, cs] { attn_backward_launch(*ap, cs); }, ap->flops_bwd, lab, ap->bytes_bwd);
    } else {
    {  // dP = go v^T ; fused: dS = scale * P * (dP - <P, dP>)
      GemmEpilogue e;
      e.out_f16 = C.dP;
      e.ldc = ldT;
      e.bs0 = ps0;
      e.bs1 = ps1;
      if (fuse_sm) {
        e.act = ACT_SOFTMAX_BWD;
        e.aux_in = ly.P;
        e.alpha = scale;
        e.n_store = ldT;
      }
      add_gemm(C.bwd, opK(C.go, Wd, T, d, Hh, os0, B, os1), opK(ly.qkv + 2 * Wd, 3 * Wd, T, d, Hh, qs0, B, qs1), T, T, d,
               e, bnS);
    }
    if (!fuse_sm) C.bwd.add(1, [=] { softmax_backward(ly.P, c->dP, B * Hh * T, T, ldT, cs); }, 0.0, "softmax_backward");
    const float scale_b = fuse_sm ? 1.f : scale;
    {  // dq = scale dS k
      GemmEpilogue e;
      e.alpha = scale_b;
      e.out_f16 = C.gqkv;
      e.ldc = 3 * Wd;
      e.bs0 = qs0;
      e.bs1 = qs1;
      add_gemm(C.bwd, opK(C.dP, ldT, T, ldT, Hh, ps0, B, ps1), opMN(ly.qkv + Wd, 3 * Wd, d, T, Hh, qs0, B, qs1), T, d, T,
               e, 64);
    }
    {  // dk = scale dS^T q
      GemmEpilogue e;
      e.alpha = scale_b;
      e.out_f16 = C.gqkv + Wd;
      e.ldc = 3 * Wd;
      e.bs0 = qs0;
      e.bs1 = qs1;
      add_gemm(C.bwd, opMN(C.dP, ldT, T, T, Hh, ps0, B, ps1), opMN(ly.qkv, 3 * Wd, d, T, Hh, qs0, B, qs1), T, d, T, e, 64);
    }
    {  // dv = P^T go
      GemmEpilogue e;
      e.out_f16 = C.gqkv + 2 * Wd;
      e.ldc = 3 * Wd;
      e.bs0 = qs0;
      e.bs1 = qs1;
      add_gemm(C.bwd, opMN(ly.P, ldT, T, T, Hh, ps0, B, ps1), opMN(C.go, Wd, d, T, Hh, os0, B, os1), T, d, T, e, 64);
    }
    }
    {  // gh = gqkv Wqkv
      GemmEpilogue e;
      e.out_f16 = C.gh;
      e.ldc = Wd;
      add_gemm(C.bwd, opK(C.gqkv, 3 * Wd, M, 3 * Wd), opMN(ly.wqkv, Wd, Wd, 3 * Wd), M, Wd, 3 * Wd, e);
    }
    C.bwd.add(1, [=] { ln_bwd(c->gh, ly.x_in, Wd, ly.stats1, ly.ln1, M, Wd, 1, c->gx, c->gx16); }, 0.0, "layernorm_backward");
  }
  {  // ln_pre backward (x = t + pos), then patch-embed dgrad on token rows 1..np of every image
    Clip* c = &C;
    C.bwd.add(1, [=] { layernorm_backward(c->gx16, c->t, Wd, c->pos, T, c->stats_pre, c->ln_pre.gamma, M, Wd, 0, c->gx, c->gx16, cs); }, 0.0, "layernorm_backward");
    GemmEpilogue e;
    e.out_f16 = C.g_patches;
    e.ldc = Kp;
    e.bs0 = (long long)np * Kp;
    add_gemm(C.bwd, opK(C.gx16 + Wd, Wd, np, Wd, B, (long long)T * Wd), opMN(C.conv1, Kp, Kp, Wd), np, Kp, Wd, e);
  }
}

void Engine::forward_clip(int i) {
  Clip& C = clip[i];
  patchify_forward(batch, range, n_local, cfg.cut_size, C.c.patch, C.Kp, C.patches, st);
  launches += 1;
  run(C.fwd);
  check_launch("clip forward");
}

// Prompt rows of every perceptor: its text prompts (one row each), then cutn rows per image prompt.  Row j carries its
// Prompt's weight / stop, the loss slot it sums into and 1 / (rows of that Prompt).
void Engine::rebuild_prompt_rows() {
  int off = (int)filters.size();  // filter losses come first in the reference's result list (pixray.py:1203-1222)
  for (int i = 0; i < cfg.n_clip; ++i) {
    Clip& C = clip[i];
    // the reference's result order per perceptor: spot prompts, spot-off prompts, prompts, image prompts (pixray.py:1283-1336)
    for (int which : {1, 0}) {
      Clip::Spot& sp = C.spot[which];
      dfree(sp.d_rows);
      dfree(sp.d_w);
      dfree(sp.d_stop);
      dfree(sp.d_inv);
      dfree(sp.d_slot);
      sp.loss_offset = off;
      if (sp.n > 0) {
        sp.d_rows = upload(sp.rows);
        sp.d_w = upload(sp.w);
        sp.d_stop = upload(sp.stop);
        sp.d_inv = upload(std::vector<float>(sp.n, 1.f));
        std::vector<int> slot(sp.n);
        for (int j = 0; j < sp.n; ++j) slot[j] = j;
        sp.d_slot = upload(slot);
        off += sp.n;
      }
    }
    const int D = C.c.out_dim, rows = C.n_text + n_img * cfg.cutn;
    std::vector<float> pr((size_t)rows * D, 0.f), w(rows), stp(rows), inv(rows);
    std::vector<int> slot(rows);
    std::copy(C.text_rows.begin(), C.text_rows.end(), pr.begin());
    for (int j = 0; j < C.n_text; ++j) {
      w[j] = C.text_w[j];
      stp[j] = C.text_stop[j];
      slot[j] = j;
      inv[j] = 1.f;
    }
    for (int k = 0; k < n_img; ++k)
      for (int r = 0; r < cfg.cutn; ++r) {
        const int j = C.n_text + k * cfg.cutn + r;
        w[j] = img_w[k];
        stp[j] = -INFINITY;  // Prompt(embed, weight) with the default stop (pixray.py:1331-1333)
        slot[j] = C.n_text + k;
        inv[j] = 1.f / cfg.cutn;
      }
    dfree(C.prompts);
    dfree(C.pweights);
    dfree(C.pstops);
    dfree(C.pinv);
    dfree(C.pslot);
    if (rows > 0) {
      C.prompts = upload(pr);
      C.pweights = upload(w);
      C.pstops = upload(stp);
      C.pinv = upload(inv);
      C.pslot = dalloc<int>(rows);
      PXR_CUDA(cudaMemcpyAsync(C.pslot, slot.data(), sizeof(int) * rows, cudaMemcpyHostToDevice, st));
      PXR_CUDA(cudaStreamSynchronize(st));
    }
    C.n_rows = rows;
    C.n_prompts = C.n_text + n_img;
    C.loss_offset = off;
    off += C.n_prompts;
  }
  if (off + (int)anchors.size() + (int)aux.size() > 64) throw EngineError(-16, "at most 64 losses (prompts + anchors + auxiliary) in total");
  total_prompts = off;
}

// The throwaway image Prompts of this iteration (pixray.py:1308-1336): make_cutouts(timg) replays the iteration's cached
// transforms (no ColorJitter on that path, pixray.py:480-486; fresh noise), perceptor.encode_image, and the [cutn, D]
// unit embeddings become the rows of Prompt(embed, weight).  Forward only: the targets are constants.  Runs before
// the main pass, which then overwrites every buffer used here.
void Engine::encode_image_prompts() {
  if (n_img == 0) return;
  const size_t ncs = (size_t)3 * src_h * src_w;
  for (int k = 0; k < n_img; ++k) {
    CutoutArgs a = cut_args;
    a.jitter = nullptr;
    a.iter = cut_args.iter + (k + 1) * (1 << 24);  // engine-drawn noise: an independent Philox stream per call
    a.pooled = img_prompts + k * ncs;
    cutout_forward(a, batch, part_min, part_max, part_imin, part_imax, st);
    minmax_reduce(nullptr, part_min, part_max, part_imin, part_imax, n_parts, range, irange, st);
    launches += 2;
    if (comm) {
      range_pack(range, xbuf, st);
      nccl_check(Comm::api().all_reduce(xbuf, xbuf, 2, Comm::kFloat32, Comm::kMin, comm, st), "allreduce(min,max)");
      range_unpack(xbuf, range, irange, st);
      launches += 3;
    }
    for (int i = 0; i < cfg.n_clip; ++i) {
      Clip& C = clip[i];
      const int D = C.c.out_dim;
      patchify_forward(batch, range, n_local, cfg.cut_size, C.c.patch, C.Kp, C.patches, st);
      run(C.fwd);
      float* rows = C.prompts + (size_t)(C.n_text + k * cfg.cutn) * D;
      if (comm) PXR_CUDA(cudaMemsetAsync(rows, 0, sizeof(float) * cfg.cutn * D, st));
      // zero prompt rows: the kernel only normalises (slip.py:66) into `rows`; de is overwritten by the main pass
      prompt_loss(C.e, C.B, D, C.prompts, C.pweights, C.pstops, C.pslot, C.pinv, 0, cfg.cutn, S,
                  rows + (size_t)first_global * D, losses_dev + C.loss_offset, C.de, C.de16, st);
      launches += 2;
      if (comm)  // every rank needs all cutn rows; each rank filled its own, the others are zero: the sum is exact
        nccl_check(Comm::api().all_reduce(rows, rows, (size_t)cfg.cutn * D, Comm::kFloat32, Comm::kSum, comm, st),
                   "allreduce(image prompt rows)");
    }
  }
  check_launch("image prompts");
}

void Engine::loss_clip(int i) {
  Clip& C = clip[i];
  if (C.n_prompts == 0) throw EngineError(-70, "no prompts set for perceptor " + std::to_string(i));
  prompt_loss(C.e, C.B, C.c.out_dim, C.prompts, C.pweights, C.pstops, C.pslot, C.pinv, C.n_rows, cfg.cutn, S, C.e_unit,
              losses_dev + C.loss_offset, C.de, C.de16, st);
  launches += 1;
  if (i == cfg.n_clip - 1 && !aux.empty()) aux_after_embed();
}

// ---- auxiliary losses.  Where each one enters the hand-written backward chain mirrors which tensor the reference
// loss reads: `globals["embeds"]` (pixray.py:1372-1376, the LAST perceptor's embeddings), `cur_cutouts`, or `out`.
void Engine::aux_after_embed() {
  for (size_t k = 0; k < aux.size(); ++k) {
    AuxLoss& a = aux[k];
    if (a.kind != PXR_LOSS_AESTHETIC) continue;
    Clip& C = clip[cfg.n_clip - 1];
    if (a.n_dev != C.c.out_dim) throw EngineError(-81, "aesthetic head width does not match the last perceptor's embedding");
    aux_aesthetic(C.e, C.B, C.c.out_dim, cfg.cutn, a.dev, a.prm[1], a.prm[0], a.weight, S, C.de, C.de16, aux_part,
                  losses_dev + aux_base() + k, st);
    launches += 2;
  }
}

void Engine::aux_on_cutouts() {
  const int cs_ = cfg.cut_size;
  for (size_t k = 0; k < aux.size(); ++k) {
    AuxLoss& a = aux[k];
    float* slot = losses_dev + aux_base() + k;
    if (a.kind == PXR_LOSS_SATURATION) {
      aux_saturation_moments(batch, n_local, cs_, aux_part, aux_sums, st);
      if (comm) nccl_check(Comm::api().all_reduce(aux_sums, aux_sums, 4, Comm::kFloat64, Comm::kSum, comm, st), "allreduce(saturation moments)");
      // the value is a function of the GLOBAL moments: one rank contributes it to the (summed) loss vector
      aux_saturation_grad(batch, n_local, cs_, cfg.cutn, aux_sums, a.weight * a.prm[0], S, cfg.rank == 0, g_batch, slot, st);
      launches += 3;
    } else if (a.kind == PXR_LOSS_PALETTE) {
      aux_palette(batch, n_local, cs_, cfg.cutn, a.dev, a.n_dev / 3, a.weight * a.prm[0], S, g_batch, aux_best, aux_part, slot, st);
      launches += 2;
    } else if (a.kind == PXR_LOSS_SMOOTHNESS) {
      if (comm) {  // torch.gradient runs over the stacked rows of ALL cutouts: two halo rows from each neighbour
        PXR_CUDA(cudaMemsetAsync(aux_xbuf, 0, sizeof(float) * 12 * cs_ * cfg.world, st));
        aux_smooth_pack_halo(batch, n_local, cs_, cfg.rank, aux_xbuf, st);
        nccl_check(Comm::api().all_reduce(aux_xbuf, aux_xbuf, (size_t)12 * cs_ * cfg.world, Comm::kFloat32, Comm::kSum, comm, st), "allreduce(smoothness halo)");
        aux_smooth_unpack_halo(aux_xbuf, cs_, cfg.rank, cfg.world, aux_halo, st);
        launches += 3;
      }
      aux_smoothness(batch, n_local, cs_, first_global, cfg.cutn, aux_halo, a.prm[2], (int)a.prm[1], a.weight * a.prm[0], S,
                     aux_A, g_batch, aux_part, slot, st);
      launches += 3;
    }
  }
}

void Engine::aux_on_image() {
  const int H = cur_cut_h(), Wd = cur_cut_w();
  const float* img = cur_cut_img();   // `out` of do_synth_and_filter: the FILTERED image (pixray.py:1384-1393)
  float* g_img = cur_g_cut_img();
  for (size_t k = 0; k < aux.size(); ++k) {
    AuxLoss& a = aux[k];
    float* slot = losses_dev + aux_base() + k;
    if (a.kind == PXR_LOSS_SYMMETRY) {
      aux_symmetry(img, H, Wd, a.weight * a.prm[0], S, g_img, aux_part, slot, st);
      launches += 2;
    } else if (a.kind == PXR_LOSS_EDGE) {
      const int m[4] = {(int)a.prm[2], (int)a.prm[3], (int)a.prm[4], (int)a.prm[5]};
      aux_edge(img, H, Wd, m, &a.prm[6], a.prm[0], a.prm[1], a.weight, S, g_img, aux_part, slot, st);
      launches += 2;
    } else if (a.kind == PXR_LOSS_GAUSSIAN) {
      aux_gaussian(img, H, Wd, a.prm[1], a.prm[2], &a.prm[3], a.weight * a.prm[0], S, g_img, aux_part, slot, st);
      launches += 2;
    }
  }
}

// CLIP backward of every participating perceptor -> d loss / d cutouts -> (range terms, ColorJitter, warp adjoint) ->
// d loss / d pooled [-> un-stretch] [-> spot mask] -> d loss / d image (= or +=).  `a` = the cutout parameters of the pass
// whose activations are live; mask_which >= 0: a spot pass (only the perceptors with spot prompts of that kind ran).
void Engine::backward_to_image(const CutoutArgs& a, int mask_which, bool accumulate_img, bool main_pass) {
  bool first = true;
  const FxPass fx_sums = next_fx(1);
  for (int i = 0; i < cfg.n_clip; ++i) {
    Clip& C = clip[i];
    if (mask_which >= 0 && C.spot[mask_which].n == 0) continue;
    run(C.bwd);
    patchify_backward(C.g_patches, batch, range, n_local, cfg.cut_size, C.c.patch, C.Kp, !first, g_batch, sums_fx, fx_sums, st);
    first = false;
    launches += 1;
  }
  if (main_pass && !aux.empty()) aux_on_cutouts();
  range_sums_finish(sums_fx, fx_sums, sums, st);  // fixed point -> fp32 (and the accumulator is clean for the next pass)
  if (comm)  // d/dmin, d/dmax terms need the sums over ALL cutouts
    nccl_check(Comm::api().all_reduce(sums, sums, 2, Comm::kFloat32, Comm::kSum, comm, st), "allreduce(sums)");
  cutout_backward(a, g_batch, range, irange, sums, grad_fx, next_fx(0), g_cut_src, st);
  launches += 2;
  const int ncs = 3 * cfg.cut_size * cfg.cut_size;
  if (aspect != 1.0) {
    rescale_bilinear_backward(g_cut_src, cfg.cut_size, cfg.cut_size, src_h, src_w, grad_fx, next_fx(0), g_pooled, st);
    launches += 2;
  }
  if (mask_which >= 0) {  // cutout[0][mask_indexes] = 0 (pixray.py:466): no gradient through the zeroed pixels
    spot_mask_apply(g_pooled, spot_mask, mask_which == 1, ncs, g_pooled, st);
    launches += 1;
  }
  pool_backward(g_pooled, pool_argmax, cur_cut_h(), cur_cut_w(), cfg.cut_size, cur_g_cut_img(), st, accumulate_img ? 1 : 0);
  launches += 2;
}

void Engine::backward_drawer() {
  if (comm) {
    // The path's one exchange step.  It sits on the IMAGE gradient, not on z.grad: ClampWithGrad's backward
    // (vqgan.py:76-79) masks by the sign of the incoming gradient, so the drawer backward is not linear in it and
    // must see the gradient of ALL cutouts.  Every rank then runs the (replicated) drawer backward on identical bits.
    Comm& c = Comm::api();
    nccl_check(c.group_start(), "group start");
    nccl_check(c.all_reduce(cur_g_cut_img(), cur_g_cut_img(), (size_t)3 * cur_cut_h() * cur_cut_w(), Comm::kFloat32, Comm::kSum,
                            comm, st),
               "allreduce(d loss / d image)");
    nccl_check(c.all_reduce(losses_dev, losses_dev, 64, Comm::kFloat32, Comm::kSum, comm, st), "allreduce(losses)");
    nccl_check(c.group_end(), "group end");
    launches += 2;
  }
  // image losses are replicated (every rank holds the same `out`): added after the exchange, values written, not summed
  if (!aux.empty()) aux_on_image();
  if (!anchors.empty()) anchors_on_image();
  if (filtered_valid) filters_backward();  // d loss / d filtered image -> d loss / d image (+ the filters' own loss gradients)
  if (cfg.drawer == PXR_DRAWER_VDIFF) vdiff_backward();
  else run(drawer_bwd);
  if (!anchors.empty()) anchors_on_z();
  check_launch("backward");
}

// init_weight_pix (pixray.py:1363-1368): l1 between `out` (the filtered image) and the init image, replicated on every rank
void Engine::anchors_on_image() {
  const long long n = 3LL * cur_cut_h() * cur_cut_w();
  for (size_t k = 0; k < anchors.size(); ++k) {
    Anchor& a = anchors[k];
    if (a.kind != PXR_ANCHOR_PIX) continue;
    if ((long long)a.n != n) throw EngineError(-82, "init_weight_pix: the init image must have the size of the (filtered) image");
    anchor_pix(cur_cut_img(), a.ref, n, a.weight, S, cur_g_cut_img(), aux_part, losses_dev + total_prompts + k, st);
    launches += 2;
  }
}

// init_weight / init_weight_dist / init_weight_cos / image_labels (pixray.py:1344-1375): terms between drawer.get_z() and
// a stored latent; their gradient never passes the drawer, so it is added to z.grad after the drawer backward
void Engine::anchors_on_z() {
  for (size_t k = 0; k < anchors.size(); ++k) {
    Anchor& a = anchors[k];
    if (a.kind == PXR_ANCHOR_PIX) continue;
    anchor_z(a.kind, z_buf, a.ref, (int)z_numel, a.weight, z_grad, losses_dev + total_prompts + k, st);
    launches += 1;
  }
}

void Engine::backward_all() {
  backward_to_image(cut_args, -1, spot_accumulated, true);
  spot_accumulated = false;
  backward_drawer();
}

// One spot pass (pixray.py:1262-1293): the pooled image with the spot (which = 1) or everything but the spot (which = 0)
// zeroed, cut with THIS iteration's cached transforms (the cached path: no ColorJitter, fresh noise, pixray.py:480-486),
// encoded by every perceptor that has spot prompts of this kind, scored, and taken back to the image gradient right away
// (the activations are single-buffered; the drawer backward runs once, on the sum, in backward_drawer).
// `pooled` must hold the current image's pooling.  Returns false when no perceptor has such prompts.
bool Engine::spot_pass(int which, bool accumulate_img) {
  if (!any_spot(which)) return false;
  if (!spot_mask) throw EngineError(-71, "spot prompts need a spot mask (pxr_set_spot_mask)");
  const int ncs = 3 * cfg.cut_size * cfg.cut_size;
  spot_mask_apply(pooled, spot_mask, which == 1, ncs, pooled_masked, st);
  CutoutArgs a = cut_args;
  a.jitter = nullptr;
  a.iter = cut_args.iter + (9 + which) * (1 << 24);  // engine-drawn noise: its own Philox stream
  if (aspect != 1.0) {
    rescale_bilinear(pooled_masked, cfg.cut_size, cfg.cut_size, src_h, src_w, cut_src, st);
    a.pooled = cut_src;
    launches += 1;
  } else {
    a.pooled = pooled_masked;
  }
  cutout_forward(a, batch, part_min, part_max, part_imin, part_imax, st);
  minmax_reduce(nullptr, part_min, part_max, part_imin, part_imax, n_parts, range, irange, st);
  launches += 3;
  if (comm) {
    range_pack(range, xbuf, st);
    nccl_check(Comm::api().all_reduce(xbuf, xbuf, 2, Comm::kFloat32, Comm::kMin, comm, st), "allreduce(min,max)");
    range_unpack(xbuf, range, irange, st);
    launches += 3;
  }
  for (int i = 0; i < cfg.n_clip; ++i) {
    Clip& C = clip[i];
    Clip::Spot& sp = C.spot[which];
    if (sp.n == 0) continue;
    forward_clip(i);
    prompt_loss(C.e, C.B, C.c.out_dim, sp.d_rows, sp.d_w, sp.d_stop, sp.d_slot, sp.d_inv, sp.n, cfg.cutn, S, C.e_unit,
                losses_dev + sp.loss_offset, C.de, C.de16, st);
    launches += 1;
  }
  backward_to_image(a, which, accumulate_img, false);
  return true;
}

void Engine::step(float lr) {
  ++adam_t;
  const int per_channel = (cfg.drawer == PXR_DRAWER_VQGAN) ? (int)(z_numel / cfg.z_channels) : 1;
  opt_clip_step(opt_kind, z_buf, OptState{adam_m, adam_v, opt_prev}, batches > 1 ? z_grad_acc : z_grad, 1.f, (int)z_numel,
                per_channel, zmin, zmax, cfg.drawer == PXR_DRAWER_PIXEL, lr, cfg.beta1, cfg.beta2, cfg.adam_eps, adam_t, st);
  launches += 1;
}

// ---- filters (kernels_filters.cu).  Every filter becomes primitives over planar [3, H, W] buffers; EDGE primitives are taps
// (loss + gradient on the tensor they look at), the others produce a new tensor.
void Engine::rebuild_filters() {
  fprims.clear();
  int H = cfg.image_h, Wd = cfg.image_w;
  const float* cur = img;
  float* cur_g = g_img;
  auto produce = [&](FilterPrim pr, int Ho, int Wo) {
    pr.Hin = H;
    pr.Win = Wd;
    pr.Hout = Ho;
    pr.Wout = Wo;
    pr.in = cur;
    pr.g_in = cur_g;
    pr.out = dalloc<float>((size_t)3 * Ho * Wo);
    pr.g_out = dalloc<float>((size_t)3 * Ho * Wo);
    fprims.push_back(pr);
    cur = pr.out;
    cur_g = pr.g_out;
    H = Ho;
    Wd = Wo;
  };
  auto tap = [&](FilterPrim pr) {
    pr.Hin = pr.Hout = H;
    pr.Win = pr.Wout = Wd;
    pr.in = cur;
    pr.g_in = cur_g;
    fprims.push_back(pr);
  };
  for (size_t f = 0; f < filters.size(); ++f) {
    Filter& F = filters[f];
    F.H = H;
    F.W = Wd;
    FilterPrim pr{};
    pr.filter = (int)f;
    if (F.kind == PXR_FILTER_TILER) {
      pr.kind = FP_ROLL;
      pr.use_h = pr.use_w = 1;
      produce(pr, H, Wd);
    } else if (F.kind == PXR_FILTER_LOOKUP) {
      pr.kind = FP_LOOKUP;
      pr.beta = F.beta;
      produce(pr, H, Wd);
    } else {  // wallpaper.py:27-93
      const int em = F.em, em2 = em / 2;
      if (F.wp_type == 1) {  // "shift"
        pr.kind = FP_WSHIFT;
        produce(pr, 2 * H, Wd);
        continue;
      }
      const bool horiz = F.wp_type == 2 || F.wp_type == 0, vert = F.wp_type == 3 || F.wp_type == 0;
      int n_edge = 0;
      if (horiz && em != 0) {
        if (em > Wd || Wd - 2 * em2 < 1 || em2 < 1) throw EngineError(-73, "wallpaper_edge_match does not fit the image width");
        FilterPrim e = pr;
        e.kind = FP_EDGE;
        e.em = em;
        e.axis = 0;
        e.accumulate = n_edge++;
        tap(e);
        FilterPrim c = pr;
        c.kind = FP_CROP;
        c.left = em2;
        produce(c, H, Wd - 2 * em2);
      }
      if (vert && em != 0) {
        if (em > H || H - 2 * em2 < 1 || em2 < 1) throw EngineError(-73, "wallpaper_edge_match does not fit the image height");
        FilterPrim e = pr;
        e.kind = FP_EDGE;
        e.em = em;
        e.axis = 1;
        e.accumulate = n_edge++;
        tap(e);
        FilterPrim c = pr;
        c.kind = FP_CROP;
        c.top = em2;
        produce(c, H - 2 * em2, Wd);
      }
      pr.kind = FP_ROLL;
      pr.use_h = vert ? 1 : 0;
      pr.use_w = horiz ? 1 : 0;
      produce(pr, H, Wd);
    }
  }
  cut_img = const_cast<float*>(cur);
  g_cut_img = cur_g;
  cut_h = H;
  cut_w = Wd;
  if (!filter_dummy) filter_dummy = dalloc<float>(4);
  if (!lookup_best) lookup_best = dalloc<int>((size_t)4 * cfg.image_h * cfg.image_w);
  rebuild_prompt_rows();
}

void Engine::filters_forward(int iter) {
  for (size_t f = 0; f < filters.size(); ++f) {
    Filter& F = filters[f];  // rand_w = torch.randint(0, W), rand_h = torch.randint(0, H), drawn by every filter call
    F.sh = F.fixed_h >= 0 ? F.fixed_h % F.H : (int)(philox_uniform(cfg.seed, (uint32_t)iter, 6u, 2 * f) * 0.999999f * F.H);
    F.sw = F.fixed_w >= 0 ? F.fixed_w % F.W : (int)(philox_uniform(cfg.seed, (uint32_t)iter, 6u, 2 * f + 1) * 0.999999f * F.W);
  }
  const float value_w = cfg.rank == 0 ? 1.f : 0.f;  // the loss vector is summed over ranks: one rank reports the replicated value
  for (FilterPrim& pr : fprims) {
    Filter& F = filters[pr.filter];
    float* slot = losses_dev + pr.filter;
    switch (pr.kind) {
      case FP_ROLL:
        filter_roll(pr.in, pr.Hin, pr.Win, pr.use_h ? F.sh % pr.Hin : 0, pr.use_w ? F.sw % pr.Win : 0, pr.out, st);
        break;
      case FP_WSHIFT: filter_wallpaper_shift(pr.in, pr.Hin, pr.Win, F.sh, F.sw, pr.out, st); break;
      case FP_CROP: filter_crop(pr.in, pr.Hin, pr.Win, pr.top, pr.left, pr.Hout, pr.Wout, pr.out, st); break;
      case FP_EDGE:
        filter_edge_match(pr.in, pr.Hin, pr.Win, pr.em, pr.axis, F.weight * value_w, 0.f, pr.accumulate, nullptr, slot, st);
        break;
      case FP_LOOKUP:
        filter_colorlookup(pr.in, pr.Hin * pr.Win, F.pal, F.n_col, pr.beta, F.weight * value_w, pr.out, lookup_best, aux_part, slot, st);
        launches += 1;
        break;
    }
    launches += 1;
  }
  filtered_valid = true;
  check_launch("filters forward");
}

void Engine::filters_backward() {
  for (int i = (int)fprims.size() - 1; i >= 0; --i) {
    FilterPrim& pr = fprims[i];
    Filter& F = filters[pr.filter];
    switch (pr.kind) {
      case FP_ROLL:
        filter_roll_backward(pr.g_out, pr.Hin, pr.Win, pr.use_h ? F.sh % pr.Hin : 0, pr.use_w ? F.sw % pr.Win : 0, 0, pr.g_in, st);
        break;
      case FP_WSHIFT: filter_wallpaper_shift_backward(pr.g_out, pr.Hin, pr.Win, F.sh, F.sw, 0, pr.g_in, st); break;
      case FP_CROP: filter_crop_backward(pr.g_out, pr.Hin, pr.Win, pr.top, pr.left, pr.Hout, pr.Wout, pr.g_in, st); break;
      case FP_EDGE:  // a tap: adds its loss gradient to the gradient of the tensor it looks at
        filter_edge_match(pr.in, pr.Hin, pr.Win, pr.em, pr.axis, F.weight, S, 0, pr.g_in, filter_dummy, st);
        break;
      case FP_LOOKUP:
        filter_colorlookup_backward(pr.g_out, pr.in, pr.out, pr.Hin * pr.Win, pr.beta, F.weight, S, 0, pr.g_in, st);
        break;
    }
    launches += 1;
  }
}

void Engine::write_initial_drop_state() {
  DropState s0{};
  s0.best_loss = 1e20f;
  s0.lr = drop_cfg.base_lr;
  PXR_CUDA(cudaMemcpyAsync(drop_state, &s0, sizeof s0, cudaMemcpyHostToDevice, st));
  PXR_CUDA(cudaMemcpyAsync(drop_state + 1, &s0, sizeof s0, cudaMemcpyHostToDevice, st));
  PXR_CUDA(cudaStreamSynchronize(st));  // s0 is a stack object
  drop_parity = 0;
  memset(const_cast<DropStatus*>(drop_status), 0, sizeof(DropStatus));
}

void Engine::zero_optimizer_state() {
  PXR_CUDA(cudaMemsetAsync(adam_m, 0, z_numel * sizeof(float), st));
  PXR_CUDA(cudaMemsetAsync(adam_v, 0, z_numel * sizeof(float), st));
  PXR_CUDA(cudaMemsetAsync(opt_prev, 0, z_numel * sizeof(float), st));
}

// opt.step() + clip_z + checkdrop + (scheduled | auto-stop) optimiser rebuild, all decided on the device
void Engine::step_managed(int iter) {
  const int per_channel = (cfg.drawer == PXR_DRAWER_VQGAN) ? (int)(z_numel / cfg.z_channels) : 1;
  const float* g = batches > 1 ? z_grad_acc : z_grad;
  opt_clip_managed(opt_kind, z_buf, OptState{adam_m, adam_v, opt_prev}, g, best_z, 1.f, (int)z_numel, per_channel, zmin,
                   zmax, cfg.drawer == PXR_DRAWER_PIXEL, cfg.beta1, cfg.beta2, cfg.adam_eps, losses_dev, num_losses(), iter,
                   drop_cfg, drop_state + drop_parity, drop_state + (drop_parity ^ 1), drop_status_dev, st);
  drop_parity ^= 1;
  launches += 1;
}

void Engine::finalize() {
  if (finalized) return;
  if (cfg.drawer == PXR_DRAWER_VQGAN) build_vqgan();
  else if (cfg.drawer == PXR_DRAWER_PIXEL) build_pixel();
  else if (cfg.drawer == PXR_DRAWER_FFT) build_fft();
  else if (cfg.drawer == PXR_DRAWER_VDIFF) build_vdiff();
  else throw EngineError(-47, "unknown drawer kind");
  adam_m = dalloc<float>(z_numel);
  adam_v = dalloc<float>(z_numel);
  opt_prev = dalloc<float>(z_numel);
  z_grad_acc = dalloc<float>(z_numel);
  best_z = dalloc<float>(z_numel);
  drop_state = dalloc<DropState>(2);
  {
    void* hp = nullptr;
    PXR_CUDA(cudaHostAlloc(&hp, sizeof(DropStatus), cudaHostAllocMapped));
    memset(hp, 0, sizeof(DropStatus));
    drop_status = static_cast<DropStatus*>(hp);
    void* dp = nullptr;
    PXR_CUDA(cudaHostGetDevicePointer(&dp, hp, 0));
    drop_status_dev = static_cast<DropStatus*>(dp);
  }
  build_cutouts();
  if (cfg.n_clip < 1 || cfg.n_clip > 2) throw EngineError(-53, "n_clip must be 1 or 2");
  for (int i = 0; i < cfg.n_clip; ++i) build_clip(i);
  losses_dev = dalloc<float>(64);
  losses_scratch = dalloc<float>(64);
  aux_part = dalloc<double>(std::max(4 * AUX_MAX_BLOCKS, n_local) + 8);
  aux_sums = dalloc<double>(4);
  aux_A = dalloc<float>(((size_t)n_local * cfg.cut_size + 2) * cfg.cut_size);
  aux_halo = dalloc<float>((size_t)12 * cfg.cut_size);
  aux_xbuf = dalloc<float>((size_t)12 * cfg.cut_size * cfg.world);
  aux_best = dalloc<int>((size_t)n_local * cfg.cut_size * cfg.cut_size);
  PXR_CUDA(cudaMallocHost((void**)&losses_host, 64 * sizeof(float)));
  PXR_CUDA(cudaStreamSynchronize(st));
  {
    const size_t npx = (size_t)3 * cfg.image_h * cfg.image_w, ncs = (size_t)3 * cfg.cut_size * cfg.cut_size;
    reg("img", img, npx * 4);
    reg("img_pre", img_pre, npx * 4);
    reg("g_img", g_img, npx * 4);
    reg("pooled", pooled, ncs * 4);
    reg("cut_src", cut_src, (size_t)3 * src_h * src_w * 4);
    reg("pool_argmax", pool_argmax, ncs * 4);
    reg("g_pooled", g_pooled, ncs * 4);
    reg("batch", batch, ncs * n_local * 4);
    reg("g_batch", g_batch, ncs * n_local * 4);
    reg("range", range, 16);
    reg("irange", irange, 16);
    reg("sums", sums, 16);
    reg("z_grad", z_grad, z_numel * 4);
    reg("z_grad_acc", z_grad_acc, z_numel * 4);
    reg("best_z", best_z, z_numel * 4);
    reg("z", z_buf, z_numel * 4);
    reg("losses", losses_dev, 64 * 4);
    if (vd_pred) {
      reg("vd_pred", vd_pred, npx * 4);
      reg("vd_v", vd_v, npx * 4);
    }
    reg("palette_best", aux_best, ncs / 3 * n_local * 4);
    reg("minv", minv_dev, (size_t)n_local * 36);
    for (int i = 0; i < cfg.n_clip; ++i) {
      Clip& C = clip[i];
      std::string p = "clip" + std::to_string(i) + ".";
      const size_t mw = (size_t)C.M * C.c.width;
      reg(p + "patches", C.patches, (size_t)C.B * C.np * C.Kp * 2);
      reg(p + "g_patches", C.g_patches, (size_t)C.B * C.np * C.Kp * 2);
      reg(p + "t", C.t, mw * 4);
      const size_t xb = stream16 ? 2 : 4;  // bytes per residual-stream element
      reg(p + "x0", C.layers[0].x_in, mw * xb);
      reg(p + "x_mid0", C.layers[0].x_mid, mw * xb);
      reg(p + "qkv0", C.layers[0].qkv, mw * 3 * 2);
      if (C.layers[0].P) reg(p + "P0", C.layers[0].P, (size_t)C.B * C.c.heads * C.T * C.ldT * 2);
      reg(p + "x_out", C.x_out, mw * xb);
      reg(p + "e", C.e, (size_t)C.B * C.c.out_dim * 4);
      reg(p + "de", C.de, (size_t)C.B * C.c.out_dim * 4);
      if (C.gx) reg(p + "gx", C.gx, mw * 4);
    }
  }
  for (auto& m : weights) m.clear();  // host copies no longer needed
  finalized = true;
}

#include "engine_vdiff.inc"

}  // namespace pxr

// ===================================================================================================== C ABI
using pxr::Engine;
using pxr::EngineError;

struct pxr_engine {
  Engine* e;
};
static thread_local std::string g_create_err;

#define PXR_TRY(h, ...)                                   \
  try {                                                   \
    __VA_ARGS__;                                          \
    return 0;                                             \
  } catch (const EngineError& ex) {                       \
    (h)->e->err = ex.what();                              \
    return ex.code;                                       \
  } catch (const std::exception& ex) {                    \
    (h)->e->err = ex.what();                              \
    return -999;                                          \
  }

extern "C" {

const char* pxr_version(void) { return "pixray_b200 0.1 (sm_100a)"; }
const char* pxr_last_error(pxr_handle h) { return h ? h->e->err.c_str() : g_create_err.c_str(); }

int pxr_create(const pxr_config* cfg, pxr_handle* out) {
  if (!cfg || !out) return -10;
  Engine* e = nullptr;
  try {
    e = new Engine(*cfg);
    e->create();
  } catch (const EngineError& ex) {
    g_create_err = ex.what();
    delete e;
    return ex.code;
  } catch (const std::exception& ex) {
    g_create_err = ex.what();
    delete e;
    return -999;
  }
  *out = new pxr_engine{e};
  return 0;
}

void pxr_destroy(pxr_handle h) {
  if (!h) return;
  delete h->e;
  delete h;
}

int pxr_load_weight(pxr_handle h, int module_id, const char* name, const float* data, const int64_t* dims, int ndim) {
  PXR_TRY(h, {
    if (module_id < 0 || module_id > 2) throw EngineError(-11, "bad module id");
    if (h->e->finalized) throw EngineError(-12, "weights cannot change after pxr_finalize");
    pxr::HostWeight w;
    w.dims.assign(dims, dims + ndim);
    w.data.resize((size_t)w.numel());
    PXR_CUDA(cudaMemcpy(w.data.data(), data, w.data.size() * sizeof(float), cudaMemcpyDefault));
    h->e->weights[module_id][name] = std::move(w);
  });
}

int pxr_finalize(pxr_handle h) { PXR_TRY(h, h->e->finalize()); }

int pxr_set_prompts(pxr_handle h, int clip_idx, const float* embeds, int n, int D, const float* weights,
                    const float* stops) {
  PXR_TRY(h, {
    Engine* e = h->e;
    if (!e->finalized) throw EngineError(-13, "call pxr_finalize first");
    if (clip_idx < 0 || clip_idx >= e->cfg.n_clip) throw EngineError(-14, "bad clip index");
    auto& C = e->clip[clip_idx];
    if (D != C.c.out_dim) throw EngineError(-15, "prompt embedding width does not match the perceptor");
    std::vector<float> pe((size_t)n * D);
    for (int j = 0; j < n; ++j) {  // F.normalize(self.embed), pixray.py:277
      double s = 0;
      for (int k = 0; k < D; ++k) s += (double)embeds[(size_t)j * D + k] * embeds[(size_t)j * D + k];
      double nrm = std::max(std::sqrt(s), 1e-12);
      for (int k = 0; k < D; ++k) pe[(size_t)j * D + k] = (float)(embeds[(size_t)j * D + k] / nrm);
    }
    C.text_rows = pe;
    C.text_w.assign(weights, weights + n);
    C.text_stop.assign(stops, stops + n);
    C.n_text = n;
    e->rebuild_prompt_rows();
  });
}

// Image prompts at their own sizes (the reference keeps each target at its aspect-preserving size, resize_image
// pixray.py:514-518, and MakeCutouts pools whatever it is given to cut_size x cut_size, pixray.py:463): imgs[k] is host or
// device fp32 [3, hs[k], ws[k]] in [0, 1].  Pooled here, once.
int pxr_set_image_prompts_sized(pxr_handle h, const float* const* imgs, const int* hs, const int* ws, int n,
                                const float* weights) {
  PXR_TRY(h, {
    Engine* e = h->e;
    if (!e->finalized) throw EngineError(-13, "call pxr_finalize first");
    if (n < 0 || (n > 0 && (!imgs || !hs || !ws))) throw EngineError(-17, "pxr_set_image_prompts: bad arguments");
    const size_t ncs = (size_t)3 * e->src_h * e->src_w;
    e->n_img = n;
    e->img_w.assign(n, 1.f);
    if (weights)
      for (int k = 0; k < n; ++k) e->img_w[k] = weights[k];
    e->dfree(e->img_prompts);
    if (n > 0) {
      e->img_prompts = e->dalloc<float>(ncs * n);
      for (int k = 0; k < n; ++k) {
        if (hs[k] < 1 || ws[k] < 1 || !imgs[k]) throw EngineError(-17, "pxr_set_image_prompts: empty image");
        float* tmp = nullptr;
        const size_t bytes = sizeof(float) * 3 * hs[k] * ws[k];
        PXR_CUDA(cudaMalloc(&tmp, bytes));
        cudaError_t ce = cudaMemcpyAsync(tmp, imgs[k], bytes, cudaMemcpyDefault, e->st);
        if (ce == cudaSuccess) {
          if (e->aspect != 1.0) {  // pooled like the canvas, then stretched like the canvas (pixray.py:463-472)
            pxr::pool_forward(tmp, hs[k], ws[k], e->cfg.cut_size, e->pooled, e->pool_argmax, e->st);
            pxr::rescale_bilinear(e->pooled, e->cfg.cut_size, e->cfg.cut_size, e->src_h, e->src_w, e->img_prompts + k * ncs, e->st);
          } else {
            pxr::pool_forward(tmp, hs[k], ws[k], e->cfg.cut_size, e->img_prompts + k * ncs, e->pool_argmax, e->st);
          }
          ce = cudaStreamSynchronize(e->st);
        }
        cudaFree(tmp);
        if (ce != cudaSuccess) throw EngineError(-200, std::string("image prompt upload failed: ") + cudaGetErrorString(ce));
      }
    }
    e->rebuild_prompt_rows();
  });
}

// Spot prompts (args.spot_prompts / args.spot_prompts_off, pixray.py:917-931, 1262-1293): which = 1 scores `embeds` on the
// cutouts of the image with the spot region zeroed (make_cutouts(out, spot=1)), which = 0 on the cutouts with everything
// BUT the spot zeroed.  n = 0 clears.  Needs pxr_set_spot_mask.  Fused path (pxr_iterate) only.
int pxr_set_spot_prompts(pxr_handle h, int clip_idx, int which, const float* embeds, int n, int D, const float* weights,
                         const float* stops) {
  PXR_TRY(h, {
    Engine* e = h->e;
    if (!e->finalized) throw EngineError(-13, "call pxr_finalize first");
    if (clip_idx < 0 || clip_idx >= e->cfg.n_clip) throw EngineError(-14, "bad clip index");
    if (which != 0 && which != 1) throw EngineError(-72, "pxr_set_spot_prompts: which = 1 (spot) or 0 (spot off)");
    auto& C = e->clip[clip_idx];
    if (n > 0 && D != C.c.out_dim) throw EngineError(-15, "prompt embedding width does not match the perceptor");
    auto& sp = C.spot[which];
    sp.rows.assign((size_t)n * (n > 0 ? D : 0), 0.f);
    for (int j = 0; j < n; ++j) {  // F.normalize(self.embed), pixray.py:277
      double s2 = 0;
      for (int k = 0; k < D; ++k) s2 += (double)embeds[(size_t)j * D + k] * embeds[(size_t)j * D + k];
      const double nrm = std::max(std::sqrt(s2), 1e-12);
      for (int k = 0; k < D; ++k) sp.rows[(size_t)j * D + k] = (float)(embeds[(size_t)j * D + k] / nrm);
    }
    sp.w.assign(weights, weights + (n > 0 ? n : 0));
    sp.stop.assign(stops, stops + (n > 0 ? n : 0));
    sp.n = n > 0 ? n : 0;
    e->rebuild_prompt_rows();
  });
}

// mask: host bytes [3, cut_size, cut_size], != 0 where the (resized, RGB) mask image is >= 0.5 (fetch_spot_indexes,
// pixray.py:370-394)
int pxr_set_spot_mask(pxr_handle h, const unsigned char* mask) {
  PXR_TRY(h, {
    Engine* e = h->e;
    if (!e->finalized) throw EngineError(-13, "call pxr_finalize first");
    if (!mask) throw EngineError(-10, "pxr_set_spot_mask: null mask");
    const size_t n = (size_t)3 * e->cfg.cut_size * e->cfg.cut_size;
    if (!e->spot_mask) e->spot_mask = e->dalloc<unsigned char>(n);
    PXR_CUDA(cudaMemcpyAsync(e->spot_mask, mask, n, cudaMemcpyHostToDevice, e->st));
    PXR_CUDA(cudaStreamSynchronize(e->st));
  });
}

int pxr_set_image_prompts(pxr_handle h, const float* imgs, int n, const float* weights) {
  if (!h) return -10;
  const int H = h->e->cfg.image_h, W = h->e->cfg.image_w;
  std::vector<const float*> ptrs(n > 0 ? n : 0);
  std::vector<int> hs(ptrs.size(), H), ws(ptrs.size(), W);
  for (size_t k = 0; k < ptrs.size(); ++k) ptrs[k] = imgs ? imgs + k * (size_t)3 * H * W : nullptr;
  return pxr_set_image_prompts_sized(h, ptrs.data(), hs.data(), ws.data(), n, weights);
}

int pxr_synth(pxr_handle h, const float* z, float* out_img) {
  PXR_TRY(h, {
    Engine* e = h->e;
    if (z) PXR_CUDA(cudaMemcpyAsync(e->z_buf, z, e->z_numel * sizeof(float), cudaMemcpyDeviceToDevice, e->st));
    e->filtered_valid = false;  // the per-op path sees the drawer's image; filters live in the fused iteration
    e->forward_drawer();
    e->check_launch("synth");
    if (out_img)
      PXR_CUDA(cudaMemcpyAsync(out_img, e->img, sizeof(float) * 3 * e->cfg.image_h * e->cfg.image_w,
                               cudaMemcpyDeviceToDevice, e->st));
  });
}

// model.encode(init_tensor)[0] (VqganDrawer.init_from_tensor / reapply_from_tensor / get_z_from_tensor, vqgan.py:174-185):
// img device fp32 [3, H, W] in [-1, 1] -> z_out device fp32 [z_channels, h, w] = the codebook rows nearest to
// quant_conv(encoder(img)).  Needs the checkpoint's encoder.* / quant_conv.* tensors (loaded before pxr_finalize).
int pxr_vqgan_encode(pxr_handle h, const float* img, float* z_out) {
  PXR_TRY(h, {
    Engine* e = h->e;
    if (e->cfg.drawer != PXR_DRAWER_VQGAN) throw EngineError(-67, "pxr_vqgan_encode: not a VQGAN engine");
    if (!e->have_encoder) throw EngineError(-67, "pxr_vqgan_encode: the loaded VQGAN weights carry no encoder.* tensors");
    if (!img || !z_out) throw EngineError(-10, "pxr_vqgan_encode: null pointer");
    PXR_CUDA(cudaMemcpyAsync(e->enc_img, img, sizeof(float) * 3 * e->cfg.image_h * e->cfg.image_w, cudaMemcpyDeviceToDevice, e->st));
    e->run(e->enc_fwd);
    e->check_launch("vqgan encode");
    PXR_CUDA(cudaMemcpyAsync(z_out, e->enc_z, sizeof(float) * e->z_numel, cudaMemcpyDeviceToDevice, e->st));
  });
}

int pxr_set_color_jitter(pxr_handle h, float p, float saturation, float hue) {
  PXR_TRY(h, {
    if (!(p >= 0.f && p <= 1.f) || saturation < 0.f || saturation > 1.f || hue < 0.f || hue > 0.5f)
      throw EngineError(-62, "pxr_set_color_jitter: p in [0,1], saturation in [0,1], hue in [0,0.5]");
    h->e->cj_p = p;
    h->e->cj_sat = saturation;
    h->e->cj_hue = hue;
  });
}

int pxr_make_cutouts(pxr_handle h, const float* img, const pxr_cut_params* p, int iter, float* out_batch) {
  PXR_TRY(h, {
    Engine* e = h->e;
    if (img) {
      PXR_CUDA(cudaMemcpyAsync(e->img, img, sizeof(float) * 3 * e->cfg.image_h * e->cfg.image_w,
                               cudaMemcpyDeviceToDevice, e->st));
      e->filtered_valid = false;
    }
    e->prepare_cut_params(p, iter);
    e->encode_image_prompts();
    e->forward_cutouts();
    if (out_batch)
      PXR_CUDA(cudaMemcpyAsync(out_batch, e->batch,
                               sizeof(float) * e->n_local * 3 * e->cfg.cut_size * e->cfg.cut_size,
                               cudaMemcpyDeviceToDevice, e->st));
  });
}

int pxr_encode_image(pxr_handle h, int clip_idx, const float* batch, float* out_embeds) {
  PXR_TRY(h, {
    Engine* e = h->e;
    if (clip_idx < 0 || clip_idx >= e->cfg.n_clip) throw EngineError(-14, "bad clip index");
    if (batch) {
      // a caller-provided batch: recompute its global range exactly like CLIP_Base.preprocess does
      PXR_CUDA(cudaMemcpyAsync(e->batch, batch, sizeof(float) * e->n_local * 3 * e->cfg.cut_size * e->cfg.cut_size,
                               cudaMemcpyDeviceToDevice, e->st));
      const int np_ = e->n_parts < 1024 ? e->n_parts : 1024;
      pxr::minmax_partials(e->batch, (long long)e->n_local * 3 * e->cfg.cut_size * e->cfg.cut_size, np_, e->part_min,
                           e->part_max, e->part_imin, e->part_imax, e->st);
      pxr::minmax_reduce(nullptr, e->part_min, e->part_max, e->part_imin, e->part_imax, np_, e->range, e->irange, e->st);
      e->launches += 2;
    }
    e->forward_clip(clip_idx);
    auto& C = e->clip[clip_idx];
    // unit-norm embeddings (slip.py:66) are produced by the loss kernel; run it when prompts exist
    if (C.n_prompts > 0) {
      PXR_CUDA(cudaMemsetAsync(e->losses_dev + C.loss_offset, 0, sizeof(float) * C.n_prompts, e->st));
      e->loss_clip(clip_idx);
    }
    if (out_embeds)
      PXR_CUDA(cudaMemcpyAsync(out_embeds, C.n_prompts > 0 ? C.e_unit : C.e, sizeof(float) * C.B * C.c.out_dim,
                               cudaMemcpyDeviceToDevice, e->st));
  });
}

int pxr_prompt_loss(pxr_handle h, int clip_idx, const float* embeds, float* out_losses) {
  PXR_TRY(h, {
    Engine* e = h->e;
    if (clip_idx < 0 || clip_idx >= e->cfg.n_clip) throw EngineError(-14, "bad clip index");
    auto& C = e->clip[clip_idx];
    if (embeds) {
      // Foreign embeddings (not the ones this engine's encode_image produced): scored as given into SCRATCH buffers --
      // the perceptor's own un-normalised embeddings and their gradient (C.e / C.de, which pxr_backward consumes together
      // with the saved ViT activations) stay what the last encode_image / prompt_loss pair left there.
      if (C.n_prompts == 0) throw EngineError(-70, "no prompts set for perceptor " + std::to_string(clip_idx));
      const size_t n = (size_t)C.B * C.c.out_dim;
      if (!C.scratch) C.scratch = e->dalloc<float>(3 * n + n);  // e | e_unit | de | de16 (fp16 in the last n floats' space)
      float *se = C.scratch, *su = C.scratch + n, *sd = C.scratch + 2 * n;
      pxr::act_t* sd16 = reinterpret_cast<pxr::act_t*>(C.scratch + 3 * n);
      float* sl = e->losses_scratch;
      PXR_CUDA(cudaMemcpyAsync(se, embeds, sizeof(float) * n, cudaMemcpyDeviceToDevice, e->st));
      PXR_CUDA(cudaMemsetAsync(sl, 0, 64 * sizeof(float), e->st));
      pxr::prompt_loss(se, C.B, C.c.out_dim, C.prompts, C.pweights, C.pstops, C.pslot, C.pinv, C.n_rows, e->cfg.cutn, e->S, su,
                       sl, sd, sd16, e->st);
      e->launches += 1;
      if (out_losses)
        PXR_CUDA(cudaMemcpyAsync(out_losses, sl, sizeof(float) * C.n_prompts, cudaMemcpyDeviceToDevice, e->st));
      return 0;
    }
    PXR_CUDA(cudaMemsetAsync(e->losses_dev + C.loss_offset, 0, sizeof(float) * C.n_prompts, e->st));
    e->loss_clip(clip_idx);
    if (out_losses)
      PXR_CUDA(cudaMemcpyAsync(out_losses, e->losses_dev + C.loss_offset, sizeof(float) * C.n_prompts,
                               cudaMemcpyDeviceToDevice, e->st));
  });
}

int pxr_backward(pxr_handle h, float* z_grad) {
  PXR_TRY(h, {
    Engine* e = h->e;
    e->backward_all();
    if (z_grad)
      PXR_CUDA(cudaMemcpyAsync(z_grad, e->z_grad, e->z_numel * sizeof(float), cudaMemcpyDeviceToDevice, e->st));
  });
}

int pxr_step(pxr_handle h, float* z, float lr, int iter) {
  PXR_TRY(h, {
    Engine* e = h->e;
    (void)iter;
    e->step(lr);
    if (z) PXR_CUDA(cudaMemcpyAsync(z, e->z_buf, e->z_numel * sizeof(float), cudaMemcpyDeviceToDevice, e->st));
  });
}

int pxr_iterate(pxr_handle h, float* z, float lr, int iter, const pxr_cut_params* p, float* out_losses_host) {
  PXR_TRY(h, {
    Engine* e = h->e;
    if (z) PXR_CUDA(cudaMemcpyAsync(e->z_buf, z, e->z_numel * sizeof(float), cudaMemcpyDeviceToDevice, e->st));
    if (e->batches > 1 && p) throw EngineError(-63, "batches > 1 draws its cutout parameters in the engine: pass p = NULL");
    e->vd_iter_request = iter;
    for (int b = 0; b < e->batches; ++b) {
      // every pass is one ascend_txt + backward (pixray.py:1464-1482): fresh augmentations, gradients accumulate in z.grad;
      // checkdrop and the reported loss vector use the FIRST pass (`if i == 0`, pixray.py:1466)
      e->rng_iter = b == 0 ? 0 : iter + b * (1 << 20);
      e->prepare_cut_params(p, iter);
      if (b == 0) PXR_CUDA(cudaMemsetAsync(e->losses_dev, 0, 64 * sizeof(float), e->st));
      else PXR_CUDA(cudaMemsetAsync(e->losses_scratch, 0, 64 * sizeof(float), e->st));
      float* keep = e->losses_dev;
      if (b > 0) e->losses_dev = e->losses_scratch;  // later passes must not disturb the first pass's loss vector
      try {
        e->encode_image_prompts();
        if (b == 0) {
          e->forward_drawer();  // same z: the image of the later passes is the same image
          if (!e->filters.empty()) e->filters_forward(iter);
        }
        if (e->any_spot(1) || e->any_spot(0)) {  // spot / spot-off prompts: their own masked cutout batches (pixray.py:1262-1293)
          pxr::pool_forward(e->cur_cut_img(), e->cur_cut_h(), e->cur_cut_w(), e->cfg.cut_size, e->pooled, e->pool_argmax, e->st);
          e->launches += 1;
          bool acc = false;
          acc |= e->spot_pass(1, acc);
          acc |= e->spot_pass(0, acc);
          e->spot_accumulated = acc;
        }
        e->forward_cutouts();
        for (int i = 0; i < e->cfg.n_clip; ++i) {
          e->forward_clip(i);
          e->loss_clip(i);
        }
        e->backward_all();
      } catch (...) {
        e->losses_dev = keep;
        e->rng_iter = 0;
        throw;
      }
      e->losses_dev = keep;
      if (e->batches > 1) {
        pxr::accumulate_f32(e->z_grad, e->z_grad_acc, e->z_numel, b > 0, e->st);
        e->launches += 1;
      }
    }
    e->rng_iter = 0;
    if (e->managed) e->step_managed(iter);
    else e->step(lr);
    if (z) PXR_CUDA(cudaMemcpyAsync(z, e->z_buf, e->z_numel * sizeof(float), cudaMemcpyDeviceToDevice, e->st));
    if (out_losses_host) {
      PXR_CUDA(cudaMemcpyAsync(e->losses_host, e->losses_dev, 64 * sizeof(float), cudaMemcpyDeviceToHost, e->st));
      PXR_CUDA(cudaStreamSynchronize(e->st));
      memcpy(out_losses_host, e->losses_host, sizeof(float) * e->num_losses());
    }
  });
}

// train()'s control decisions on the device (checkdrop, scheduled learning-rate drops, auto-stop; pixray.py:1090-1109,
// 1464-1512).  After this call pxr_iterate ignores its `lr` argument: the engine owns the learning rate, the Adam step
// counter and the drop bookkeeping, and pxr_poll_status reports them without synchronising.  n_drops <= 16.
int pxr_set_schedule(pxr_handle h, float base_lr, int iter_drop_delay, int max_loss_drops, int auto_stop, const int* drops,
                     int n_drops) {
  PXR_TRY(h, {
    Engine* e = h->e;
    if (!e->finalized) throw EngineError(-13, "call pxr_finalize first");
    if (n_drops < 0 || n_drops > 16 || (n_drops > 0 && !drops)) throw EngineError(-64, "pxr_set_schedule: at most 16 scheduled drops");
    if (!(base_lr > 0.f) || iter_drop_delay < 0 || max_loss_drops < 0) throw EngineError(-64, "pxr_set_schedule: bad arguments");
    e->drop_cfg.base_lr = base_lr;
    e->drop_cfg.iter_drop_delay = iter_drop_delay;
    e->drop_cfg.max_loss_drops = max_loss_drops;
    e->drop_cfg.auto_stop = auto_stop ? 1 : 0;
    e->drop_cfg.n_sched = n_drops;
    for (int i = 0; i < n_drops; ++i) e->drop_cfg.sched[i] = drops[i];
    e->managed = true;
    e->zero_optimizer_state();
    e->write_initial_drop_state();
  });
}

// Non-blocking: the record the last COMPLETED iteration left in pinned memory.  Returns 1 when there is no consistent
// record yet (no managed iteration has finished, or the kernel is mid-write: poll again), 0 on success.
int pxr_poll_status(pxr_handle h, pxr_status* out) {
  pxr::DropStatus* s = h->e->drop_status;
  if (!s || !out) return -10;
  const int e1 = s->seq_end;
  std::atomic_thread_fence(std::memory_order_acquire);
  pxr_status r;
  r.iter = s->iter;
  r.loss_sum = s->loss_sum;
  r.best_loss = s->best_loss;
  r.best_iter = s->best_iter;
  r.num_loss_drop = s->num_loss_drop;
  r.stopped = s->stopped;
  r.rebuilt = s->rebuilt;
  r.lr = s->lr;
  r.n_losses = s->n_losses;
  for (int k = 0; k < 64; ++k) r.losses[k] = s->losses[k];
  std::atomic_thread_fence(std::memory_order_acquire);
  const int e0 = s->seq_begin;
  if (e1 == 0 || e0 != e1) return 1;
  *out = r;
  return 0;
}

int pxr_set_batches(pxr_handle h, int batches) {
  PXR_TRY(h, {
    if (batches < 1 || batches > 64) throw EngineError(-65, "batches must be in [1, 64]");
    h->e->batches = batches;
  });
}

// z.grad for the next pxr_step from the caller (the plugin loop accumulates the gradients of several passes itself)
int pxr_set_z_grad(pxr_handle h, const float* z_grad) {
  PXR_TRY(h, {
    Engine* e = h->e;
    if (!z_grad) throw EngineError(-10, "pxr_set_z_grad: null gradient");
    PXR_CUDA(cudaMemcpyAsync(e->z_grad, z_grad, e->z_numel * sizeof(float), cudaMemcpyDeviceToDevice, e->st));
  });
}

// One full iteration with a CUDA-event pair around every op (engine stream).  out[0] = ms in gemm_tc_kernel launches,
// out[1] = number of those launches, out[2] = their algorithmic FLOPs, out[3] = ms in all other kernels,
// out[4] = number of other launches, out[5] = ms of the whole iteration (first event -> last event).
int pxr_profile_iteration(pxr_handle h, float* z, float lr, int iter, double* out6) {
  return pxr_profile_iteration2(h, z, lr, iter, out6, nullptr);
}

int pxr_profile_iteration2(pxr_handle h, float* z, float lr, int iter, double* out6, double* tensor_bytes) {
  PXR_TRY(h, {
    Engine* e = h->e;
    if (z) PXR_CUDA(cudaMemcpyAsync(e->z_buf, z, e->z_numel * sizeof(float), cudaMemcpyDeviceToDevice, e->st));
    e->prepare_cut_params(nullptr, iter);
    PXR_CUDA(cudaMemsetAsync(e->losses_dev, 0, 64 * sizeof(float), e->st));
    e->prof.clear();
    e->profiling = true;
    cudaEvent_t t0;
    cudaEvent_t t1;
    PXR_CUDA(cudaEventCreate(&t0));
    PXR_CUDA(cudaEventCreate(&t1));
    PXR_CUDA(cudaEventRecord(t0, e->st));
    e->forward_drawer();
    e->forward_cutouts();
    for (int i = 0; i < e->cfg.n_clip; ++i) {
      e->forward_clip(i);
      e->loss_clip(i);
    }
    e->backward_all();
    e->step(lr);
    PXR_CUDA(cudaEventRecord(t1, e->st));
    e->profiling = false;
    PXR_CUDA(cudaStreamSynchronize(e->st));
    for (int i = 0; i < 6; ++i) out6[i] = 0;
    double tb = 0;
    FILE* dump = nullptr;
    if (const char* path = getenv("PXR_PROFILE_DUMP")) dump = fopen(path, "w");
    if (dump) fprintf(dump, "op,ms,gflop,launches\n");
    for (auto& r : e->prof) {
      float ms = 0;
      PXR_CUDA(cudaEventElapsedTime(&ms, r.a, r.b));
      if (dump) fprintf(dump, "%s,%.4f,%.3f,%d\n", r.name.empty() ? "op" : r.name.c_str(), ms, r.flops * 1e-9, r.launches);
      if (r.flops > 0) {
        out6[0] += ms;
        out6[1] += r.launches;
        out6[2] += r.flops;
        tb += r.bytes;
      } else {
        out6[3] += ms;
        out6[4] += r.launches;
      }
      cudaEventDestroy(r.a);
      cudaEventDestroy(r.b);
    }
    e->prof.clear();
    if (dump) fclose(dump);
    float tot = 0;
    PXR_CUDA(cudaEventElapsedTime(&tot, t0, t1));
    out6[5] = tot;
    if (tensor_bytes) *tensor_bytes = tb;
    cudaEventDestroy(t0);
    cudaEventDestroy(t1);
    if (z) PXR_CUDA(cudaMemcpyAsync(z, e->z_buf, e->z_numel * sizeof(float), cudaMemcpyDeviceToDevice, e->st));
  });
}

int pxr_vdiff_set_schedule(pxr_handle h, const float* steps, const float* alphas, const float* sigmas, int n) {
  PXR_TRY(h, {
    Engine* e = h->e;
    if (e->cfg.drawer != PXR_DRAWER_VDIFF) throw EngineError(-59, "not a vdiff engine");
    if (n < 1 || !steps || !alphas || !sigmas) throw EngineError(-59, "pxr_vdiff_set_schedule: empty schedule");
    e->vd_steps.assign(steps, steps + n);
    e->vd_alphas.assign(alphas, alphas + n);
    e->vd_sigmas.assign(sigmas, sigmas + n);
  });
}

int pxr_vdiff_set_clip_embed(pxr_handle h, const float* embed, int D) {
  PXR_TRY(h, {
    Engine* e = h->e;
    if (e->cfg.drawer != PXR_DRAWER_VDIFF || !e->finalized) throw EngineError(-59, "not a finalized vdiff engine");
    if (D != 512) throw EngineError(-59, "cc12m_1 is conditioned on a 512-wide CLIP embedding");
    // cc12m_1.py:244: F.normalize(clip_embed) * sqrt(D)
    std::vector<float> ce(embed, embed + D);
    double s = 0;
    for (float v : ce) s += (double)v * v;
    const double k = std::sqrt((double)D) / std::max(std::sqrt(s), 1e-12);
    for (float& v : ce) v = (float)(v * k);
    PXR_CUDA(cudaMemcpyAsync(e->vd_h0, ce.data(), sizeof(float) * D, cudaMemcpyHostToDevice, e->st));
    PXR_CUDA(cudaStreamSynchronize(e->st));
    e->vd_have_embed = true;
  });
}

int pxr_vdiff_set_iteration(pxr_handle h, int i) {
  h->e->vd_iter_request = i;
  return 0;
}

int pxr_vdiff_renoise(pxr_handle h, float* z, int i, const float* noise) {
  PXR_TRY(h, {
    Engine* e = h->e;
    if (e->cfg.drawer != PXR_DRAWER_VDIFF) throw EngineError(-59, "not a vdiff engine");
    const int n = (int)e->vd_steps.size();
    if (i < 0 || i >= n) throw EngineError(-59, "pxr_vdiff_renoise: iteration outside the schedule");
    if (z) PXR_CUDA(cudaMemcpyAsync(e->z_buf, z, e->z_numel * sizeof(float), cudaMemcpyDeviceToDevice, e->st));
    if (i < n - 1) {  // sampling.py:24-37 with eta = 1
      const double a = e->vd_alphas[i], s = e->vd_sigmas[i], a1 = e->vd_alphas[i + 1], s1 = e->vd_sigmas[i + 1];
      const double ddim = std::sqrt(s1 * s1 / (s * s)) * std::sqrt(std::max(0.0, 1.0 - a * a / (a1 * a1)));
      const double adj = std::sqrt(std::max(0.0, s1 * s1 - ddim * ddim));
      pxr::vd_renoise(e->z_buf, e->vd_pred, e->vd_v, noise, (float)a, (float)s, (float)a1, (float)adj, (float)ddim,
                      e->z_numel, e->st);
      e->launches += 1;
    }
    if (z) PXR_CUDA(cudaMemcpyAsync(z, e->z_buf, e->z_numel * sizeof(float), cudaMemcpyDeviceToDevice, e->st));
  });
}

int pxr_add_aux_loss(pxr_handle h, int kind, float weight, const float* params, int n_params) {
  PXR_TRY(h, {
    Engine* e = h->e;
    if (!e->finalized) throw EngineError(-13, "call pxr_finalize first");
    if (e->num_losses() >= 64) throw EngineError(-16, "at most 64 losses (prompts + auxiliary) in total");
    auto need = [&](int n, const char* what) {
      if (n_params < n || !params) throw EngineError(-80, std::string("pxr_add_aux_loss: ") + what);
    };
    Engine::AuxLoss a;
    a.kind = kind;
    a.weight = weight;
    a.prm.assign(params, params + (n_params > 0 ? n_params : 0));
    switch (kind) {
      case PXR_LOSS_SYMMETRY: need(1, "symmetry needs {symmetry_weight}"); break;
      case PXR_LOSS_SATURATION: need(1, "saturation needs {saturation_weight}"); break;
      case PXR_LOSS_PALETTE:
        need(4, "palette needs {palette_weight, r,g,b, ...}");
        if ((n_params - 1) % 3) throw EngineError(-80, "pxr_add_aux_loss: palette colours come as r,g,b triples");
        a.dev = e->upload(std::vector<float>(params + 1, params + n_params));
        a.n_dev = n_params - 1;
        break;
      case PXR_LOSS_SMOOTHNESS:
        need(3, "smoothness needs {smoothness_weight, type, spacing}");
        if (params[1] < 0 || params[1] > 2 || params[2] <= 0) throw EngineError(-80, "pxr_add_aux_loss: smoothness type in {0,1,2}, spacing > 0");
        break;
      case PXR_LOSS_EDGE: need(9, "edge needs {edge_color_weight, global_color_weight, left,right,upper,lower, r,g,b}"); break;
      case PXR_LOSS_GAUSSIAN:
        need(6, "gaussian needs {gaussian_weight, std_y, std_x, R,G,B}");
        if (params[1] <= 0 || params[2] <= 0) throw EngineError(-80, "pxr_add_aux_loss: gaussian std must be positive");
        break;
      case PXR_LOSS_AESTHETIC:
        need(3, "aesthetic needs {target, bias, w[D]}");
        a.dev = e->upload(std::vector<float>(params + 2, params + n_params));
        a.n_dev = n_params - 2;
        break;
      default: throw EngineError(-80, "pxr_add_aux_loss: unknown loss kind");
    }
    e->aux.push_back(std::move(a));
  });
}

// Filters (args.filters = "name:weight,...", pixray.py:651-668; applied to drawer.synth's output before MakeCutouts,
// pixray.py:1203-1222).  params (host floats) by kind:
//   TILER     {}                                                       filters/tiler.py: torch.roll by random (h, w) shifts
//   WALLPAPER {type (0 none, 1 shift, 2 horizontal, 3 vertical), edge_match}   filters/wallpaper.py
//   LOOKUP    {lookup_beta, r0,g0,b0, r1,g1,b1, ...} palette in [0,1]   filters/colorlookup.py
// Each filter owns one entry at the FRONT of the loss vector (0 for the loss-free ones), in the order added.
int pxr_add_filter(pxr_handle h, int kind, float weight, const float* params, int n_params) {
  PXR_TRY(h, {
    Engine* e = h->e;
    if (!e->finalized) throw EngineError(-13, "call pxr_finalize first");
    if (e->num_losses() >= 64) throw EngineError(-16, "at most 64 losses (filters + prompts + auxiliary) in total");
    Engine::Filter F{};
    F.kind = kind;
    F.weight = weight;
    if (kind == PXR_FILTER_TILER) {
    } else if (kind == PXR_FILTER_WALLPAPER) {
      if (n_params < 2 || !params) throw EngineError(-74, "wallpaper needs {type, edge_match}");
      F.wp_type = (int)params[0];
      F.em = (int)params[1];
      if (F.wp_type < 0 || F.wp_type > 3 || F.em < 0) throw EngineError(-74, "wallpaper: type in 0..3, edge_match >= 0");
    } else if (kind == PXR_FILTER_LOOKUP) {
      if (n_params < 4 || !params || (n_params - 1) % 3) throw EngineError(-74, "lookup needs {lookup_beta, r,g,b, ...}");
      F.beta = params[0];
      F.pal = e->upload(std::vector<float>(params + 1, params + n_params));
      F.n_col = (n_params - 1) / 3;
    } else {
      throw EngineError(-74, "pxr_add_filter: unknown filter kind");
    }
    e->filters.push_back(F);
    try {
      e->rebuild_filters();
    } catch (...) {
      e->filters.pop_back();
      e->rebuild_filters();
      throw;
    }
  });
}

int pxr_clear_filters(pxr_handle h) {
  PXR_TRY(h, {
    h->e->filters.clear();
    h->e->filtered_valid = false;
    h->e->rebuild_filters();
  });
}

// Explicit (rand_h, rand_w) of one filter for replays / parity tests; negative = engine-drawn again.
int pxr_set_filter_shifts(pxr_handle h, int filter_idx, int rand_h, int rand_w) {
  PXR_TRY(h, {
    Engine* e = h->e;
    if (filter_idx < 0 || filter_idx >= (int)e->filters.size()) throw EngineError(-74, "pxr_set_filter_shifts: bad filter index");
    e->filters[filter_idx].fixed_h = rand_h;
    e->filters[filter_idx].fixed_w = rand_w;
  });
}

int pxr_add_anchor(pxr_handle h, int kind, float weight, const float* ref, long long n) {
  PXR_TRY(h, {
    Engine* e = h->e;
    if (!e->finalized) throw EngineError(-13, "call pxr_finalize first");
    if (kind < PXR_ANCHOR_SPHERICAL || kind > PXR_ANCHOR_PIX) throw EngineError(-82, "pxr_add_anchor: unknown kind");
    if (!ref) throw EngineError(-82, "pxr_add_anchor: null reference");
    const long long want = kind == PXR_ANCHOR_PIX ? n : (long long)e->z_numel;
    if (n != want || n <= 0) throw EngineError(-82, "pxr_add_anchor: a latent anchor has the latent's element count");
    if (e->num_losses() + 1 > 64) throw EngineError(-16, "at most 64 losses (prompts + anchors + auxiliary) in total");
    Engine::Anchor a;
    a.kind = kind;
    a.weight = weight;
    a.n = (size_t)n;
    a.ref = e->dalloc<float>(a.n);
    PXR_CUDA(cudaMemcpyAsync(a.ref, ref, sizeof(float) * a.n, cudaMemcpyDefault, e->st));
    PXR_CUDA(cudaStreamSynchronize(e->st));
    e->anchors.push_back(a);
  });
}

int pxr_clear_anchors(pxr_handle h) {
  PXR_TRY(h, {
    for (auto& a : h->e->anchors) h->e->dfree(a.ref);
    h->e->anchors.clear();
  });
}

int pxr_clear_aux_losses(pxr_handle h) {
  PXR_TRY(h, h->e->aux.clear());
}

int pxr_num_losses(pxr_handle h, int* out) {
  *out = h->e->num_losses();
  return 0;
}

int pxr_read_losses(pxr_handle h, float* out_host) {
  PXR_TRY(h, {
    Engine* e = h->e;
    PXR_CUDA(cudaMemcpyAsync(e->losses_host, e->losses_dev, 64 * sizeof(float), cudaMemcpyDeviceToHost, e->st));
    PXR_CUDA(cudaStreamSynchronize(e->st));
    memcpy(out_host, e->losses_host, sizeof(float) * e->num_losses());
  });
}

int pxr_reset_optimizer(pxr_handle h) {
  PXR_TRY(h, {
    Engine* e = h->e;
    e->zero_optimizer_state();
    e->adam_t = 0;
    if (e->managed) e->write_initial_drop_state();  // a fresh session: best-loss tracking and the drop count restart too
  });
}

int pxr_set_optimizer(pxr_handle h, int kind) {
  if (kind < 0 || kind >= pxr::OPT_KINDS) {
    h->e->err = "pxr_set_optimizer: unknown optimiser kind " + std::to_string(kind);
    return -75;
  }
  h->e->opt_kind = kind;
  return pxr_reset_optimizer(h);
}

// ---- checkpoint of the optimisation state (z, optimiser state / kind / step, the drop bookkeeping): resume = load + keep
// iterating
namespace {
struct StateHeader {
  uint32_t magic, version;
  int64_t z_numel;
  int32_t adam_t, managed, drop_parity;
  int32_t opt_kind;  // PXR_OPT_*; 0 (Adam) in blobs written before the engine had other optimisers
  pxr::DropState drop;
};
constexpr uint32_t kStateMagic = 0x50585253u;  // "PXRS"
const char* const kOptNames[pxr::OPT_KINDS] = {"Adam", "AdamW", "Adagrad", "Adamax", "DiffGrad"};
// z, s0, s1, and s2 only for DiffGrad: an Adam blob keeps the size and layout it always had
int state_buffers(int kind) { return kind == pxr::OPT_DIFFGRAD ? 4 : 3; }
const char* opt_name(int kind) { return kind >= 0 && kind < pxr::OPT_KINDS ? kOptNames[kind] : "unknown"; }
}  // namespace

int pxr_state_size(pxr_handle h, int64_t* nbytes) {
  *nbytes = (int64_t)sizeof(StateHeader) + state_buffers(h->e->opt_kind) * h->e->z_numel * (int64_t)sizeof(float);
  return 0;
}

// host buffer of pxr_state_size bytes <- {header, z, s0, s1[, s2]}.  Blocking.
int pxr_save_state(pxr_handle h, void* host_buf) {
  PXR_TRY(h, {
    Engine* e = h->e;
    if (!host_buf) throw EngineError(-10, "pxr_save_state: null buffer");
    StateHeader hd{};
    hd.magic = kStateMagic;
    hd.version = 1;
    hd.z_numel = e->z_numel;
    hd.adam_t = e->adam_t;
    hd.managed = e->managed ? 1 : 0;
    hd.drop_parity = e->drop_parity;
    hd.opt_kind = e->opt_kind;
    if (e->managed)
      PXR_CUDA(cudaMemcpyAsync(&hd.drop, e->drop_state + e->drop_parity, sizeof(pxr::DropState), cudaMemcpyDeviceToHost, e->st));
    char* out = static_cast<char*>(host_buf);
    const size_t zb = (size_t)e->z_numel * sizeof(float);
    PXR_CUDA(cudaMemcpyAsync(out + sizeof hd, e->z_buf, zb, cudaMemcpyDeviceToHost, e->st));
    PXR_CUDA(cudaMemcpyAsync(out + sizeof hd + zb, e->adam_m, zb, cudaMemcpyDeviceToHost, e->st));
    PXR_CUDA(cudaMemcpyAsync(out + sizeof hd + 2 * zb, e->adam_v, zb, cudaMemcpyDeviceToHost, e->st));
    if (state_buffers(e->opt_kind) > 3)
      PXR_CUDA(cudaMemcpyAsync(out + sizeof hd + 3 * zb, e->opt_prev, zb, cudaMemcpyDeviceToHost, e->st));
    PXR_CUDA(cudaStreamSynchronize(e->st));
    memcpy(out, &hd, sizeof hd);
  });
}

// The inverse: the engine's z, optimiser state (the blob's optimiser kind must be the engine's) and (when it was saved in
// managed mode and pxr_set_schedule was called here too) the learning-rate / best-loss / drop-count bookkeeping.  Blocking.
int pxr_load_state(pxr_handle h, const void* host_buf) {
  PXR_TRY(h, {
    Engine* e = h->e;
    if (!host_buf) throw EngineError(-10, "pxr_load_state: null buffer");
    StateHeader hd;
    memcpy(&hd, host_buf, sizeof hd);
    if (hd.magic != kStateMagic || hd.version != 1) throw EngineError(-68, "pxr_load_state: not a pixray_b200 state blob");
    if (hd.z_numel != e->z_numel) throw EngineError(-68, "pxr_load_state: the blob belongs to a different latent shape");
    if (hd.opt_kind != e->opt_kind)
      throw EngineError(-68, std::string("pxr_load_state: the blob holds ") + opt_name(hd.opt_kind) +
                                 " state but the engine's optimiser is " + opt_name(e->opt_kind) + " (pxr_set_optimizer first)");
    const char* in = static_cast<const char*>(host_buf);
    const size_t zb = (size_t)e->z_numel * sizeof(float);
    PXR_CUDA(cudaMemcpyAsync(e->z_buf, in + sizeof hd, zb, cudaMemcpyHostToDevice, e->st));
    PXR_CUDA(cudaMemcpyAsync(e->adam_m, in + sizeof hd + zb, zb, cudaMemcpyHostToDevice, e->st));
    PXR_CUDA(cudaMemcpyAsync(e->adam_v, in + sizeof hd + 2 * zb, zb, cudaMemcpyHostToDevice, e->st));
    if (state_buffers(e->opt_kind) > 3)
      PXR_CUDA(cudaMemcpyAsync(e->opt_prev, in + sizeof hd + 3 * zb, zb, cudaMemcpyHostToDevice, e->st));
    e->adam_t = hd.adam_t;
    if (hd.managed && e->managed) {
      PXR_CUDA(cudaMemcpyAsync(e->drop_state + e->drop_parity, &hd.drop, sizeof(pxr::DropState), cudaMemcpyHostToDevice, e->st));
    }
    PXR_CUDA(cudaStreamSynchronize(e->st));
  });
}

int pxr_sync(pxr_handle h) { PXR_TRY(h, PXR_CUDA(cudaStreamSynchronize(h->e->st))); }

int pxr_num_kernel_launches(pxr_handle h, int64_t* out) {
  *out = h->e->launches;
  return 0;
}
int pxr_get_stream(pxr_handle h, void** out) {
  *out = h->e->st;
  return 0;
}
int pxr_z_numel(pxr_handle h, int64_t* out) {
  *out = h->e->z_numel;
  return 0;
}
int pxr_z_bounds(pxr_handle h, float* zmin, float* zmax) {
  PXR_TRY(h, {
    Engine* e = h->e;
    if (!e->zmin) throw EngineError(-18, "this drawer has no per-channel z bounds");
    PXR_CUDA(cudaMemcpyAsync(zmin, e->zmin, sizeof(float) * e->cfg.z_channels, cudaMemcpyDeviceToDevice, e->st));
    PXR_CUDA(cudaMemcpyAsync(zmax, e->zmax, sizeof(float) * e->cfg.z_channels, cudaMemcpyDeviceToDevice, e->st));
  });
}

int pxr_debug_read(pxr_handle h, const char* name, void* out, int64_t nbytes) {
  PXR_TRY(h, {
    Engine* e = h->e;
    auto it = e->dbg.find(name);
    if (it == e->dbg.end()) throw EngineError(-19, std::string("unknown debug buffer ") + name);
    if ((size_t)nbytes > it->second.second) throw EngineError(-19, "debug read larger than the buffer");
    PXR_CUDA(cudaMemcpyAsync(out, it->second.first, nbytes, cudaMemcpyDefault, e->st));
    PXR_CUDA(cudaStreamSynchronize(e->st));
  });
}

int pxr_set_comm(pxr_handle h, const void* nccl_unique_id, int rank, int world) {
  PXR_TRY(h, {
    Engine* e = h->e;
    if (world != e->cfg.world || rank != e->cfg.rank)
      throw EngineError(-92, "pxr_set_comm: rank/world differ from the pxr_config the engine was created with");
    if (world == 1) return 0;
    std::string msg;
    if (!pxr::Comm::api().load(&msg)) throw EngineError(-90, msg);
    pxr::NcclUniqueId id;
    memcpy(&id, nccl_unique_id, sizeof id);
    e->nccl_check(pxr::Comm::api().init_rank(&e->comm, world, id, rank), "ncclCommInitRank");
  });
}
int pxr_get_unique_id(void* out128) {
  std::string msg;
  if (!pxr::Comm::api().load(&msg)) {
    g_create_err = msg;
    return -90;
  }
  pxr::NcclUniqueId id;
  if (pxr::Comm::api().get_unique_id(&id) != 0) {
    g_create_err = "ncclGetUniqueId failed";
    return -91;
  }
  memcpy(out128, &id, sizeof id);
  return 0;
}

}  // extern "C"
