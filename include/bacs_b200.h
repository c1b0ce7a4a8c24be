/* bacs_b200.h -- C ABI of libbacs_b200.so: the BACS per-pixel continual-learning loss path
 * as hand-written sm_100a CUDA kernels.
 *
 * The upstream reference (mostafaelaraby/BACS-Continual-Semantic-Segmentation) is pure
 * Python and has no FFI for this path; its boundary is the loss-class interface
 * (SURVEY.md 8b).  The entry points below are what a binding of that interface needs;
 * each one cites the reference code it replaces (paths relative to the reference root).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - the caller owns and allocates all memory, including workspaces;
 *   - every call is asynchronous on `stream`, never synchronises, never allocates;
 *   - returns BACS_OK (0) or a negative bacs_status; bacs_last_error_string() describes
 *     the last failure on the calling thread;
 *   - tensors are dense NCHW / NHW row-major; `dtype` says how logits / features are
 *     stored (accumulation is always fp32 or fp64);
 *   - labels are int64 as the reference delivers them (base_loss.py:274-282).
 */
#ifndef BACS_B200_H_
#define BACS_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* bacs_stream_t; /* cudaStream_t */

enum bacs_status {
  BACS_OK = 0,
  BACS_ERR_INVALID = -1,     /* bad argument (shape, dtype, null pointer) */
  BACS_ERR_UNSUPPORTED = -2, /* valid request this build cannot serve */
  BACS_ERR_CUDA = -3,        /* a CUDA runtime call failed (see last error string) */
  BACS_ERR_WORKSPACE = -4    /* workspace too small */
};

enum bacs_dtype { BACS_F32 = 0, BACS_BF16 = 1, BACS_F16 = 2 };

/* Largest task count T of the task down-sample, the prototype sums and update, the peer all-reduce's prototype update
 * and bacs_seen_logits_many: the range of the int8 task map (ids 0..127, -1 = no task).  bacs_seen_logits and
 * bacs_seen_logits_heads take at most 32 heads. */
#define BACS_MAX_TASKS 128

int bacs_version(void);
const char* bacs_last_error_string(void);
/* number of SMs of the current device (grid sizing by the host side) */
int bacs_device_sm_count(void);
/* kernels launched by this library in this process so far (bench.py's gpu_launches) */
unsigned long long bacs_launch_count(void);

/* ---------------------------------------------------------------------------------
 * Labels
 * --------------------------------------------------------------------------------- */

/* hist[v] += #pixels with label v for v in [0,256); hist[256] += #labels outside [0,256).
 * Caller zeroes hist (int64[257]).  Used as the class-weighted CE normaliser
 * (F.cross_entropy weight=..., base_loss.py:237-240) and for "labels present". */
int bacs_label_hist(const int64_t* labels, int64_t n, int64_t* hist, bacs_stream_t stream);

/* Continual-learning label remap with the reference's sequential in-place semantics
 * (training/utils.py:225-261 TransformLabel; dataset/cityscape_dataset.py:77-108).
 * Two passes (id->trainId map, then the CL map); each pass visits the labels present at
 * entry in ascending order and rewrites the pixels equal to each, so chains such as
 * 3->5 then 5->2 alias exactly as in the reference (SURVEY Q13).
 * Value domain [lo, lo+n_dom), n_dom <= 1024 (Cityscapes raw ids start at -1).
 * map1/map2: int32[n_dom], entry v-lo = new value of v, unmapped entries already set to
 * that pass's masking value by the host; all map and masking values must lie inside the
 * domain.  map2 may be NULL (single pass).  Labels outside the domain behave like
 * unmapped ones.  The remap is per image (`n_images` x `pixels_per_image`) because the
 * reference transforms one target at a time.  in/out int64, may alias.
 * workspace: bacs_label_remap_workspace_bytes(n_images). */
size_t bacs_label_remap_workspace_bytes(int64_t n_images);
int bacs_label_remap(const int64_t* in, int64_t* out, int64_t n_images, int64_t pixels_per_image,
                     int lo, int n_dom, const int32_t* map1, int masking1, const int32_t* map2,
                     int masking2, int32_t* workspace, bacs_stream_t stream);

/* Nearest down-sample of the label map to the feature grid + class->task assignment +
 * per-image raster rank of every masked pixel inside its task.
 *   loss/prototypes.py:177-205 (F.interpolate nearest on the .double() mask),
 *   loss/base_loss.py:98-107  (np.rint half-to-even class->task; done on the host into
 *                              task_lut: int32[256], -1 = background / ignore / unseen)
 * outputs: labels_down int64[B,h,w] (may be NULL), task int8[B,h,w] (-1 none),
 *          rank int32[B,h,w], n_bt int32[B,T] masked pixels per image and task. */
int bacs_label_downsample_task(const int64_t* labels, int B, int H, int W, int h, int w,
                               const int32_t* task_lut, int T, int64_t* labels_down,
                               int8_t* task, int32_t* rank, int32_t* n_bt,
                               bacs_stream_t stream);

/* ---------------------------------------------------------------------------------
 * Prototypes (loss/prototypes.py:127-163, 31-40)
 * --------------------------------------------------------------------------------- */

/* Segmented reduction of label-masked features into per-task sums.
 * mode 0 = reference-exact: reproduces features[mask.expand(..)].view(D,-1).sum(-1),
 *          whose rows are NOT channels when B > 1 (SURVEY Q1);
 * mode 1 = per-channel sums (what the reference computes when B == 1; decomposable
 *          across ranks).
 * sums fp64[T,D] and counts fp64[T] are OVERWRITTEN (fp64 so that the packed all-reduce
 * of sums|counts is exact for counts).  workspace >= bacs_proto_workspace_bytes.
 * 16-bit features with h*w a multiple of 32 and D a multiple of 16 run as a one-hot GEMM on the
 * tensor cores whose per-(image, channel, task) totals are added into sums with fp64 atomics
 * (exact, hence order-independent, unless the ~B fp32-valued addends of a row span more than
 * 29 binary orders of magnitude); other inputs use the shared-memory-table kernel and a gather
 * pass in a fixed order. */
size_t bacs_proto_workspace_bytes(int B, int D, int T);
int bacs_proto_accumulate(const void* features, int dtype, int B, int D, int h, int w,
                          const int8_t* task, const int32_t* rank, const int32_t* n_bt, int T,
                          int mode, double* sums, double* counts, void* workspace,
                          size_t workspace_bytes, bacs_stream_t stream);

/* bacs_proto_accumulate followed by bacs_proto_update in the same two launches (single-process training step: no
 * exchange between the sums and the update; prototypes.py:127-163).  sums / counts are still written. */
int bacs_proto_accumulate_update(const void* features, int dtype, int B, int D, int h, int w,
                                 const int8_t* task, const int32_t* rank, const int32_t* n_bt, int T,
                                 int mode, double* sums, double* counts, void* workspace,
                                 size_t workspace_bytes, float* proto, void* count, int count_is_int64,
                                 int32_t* ready, bacs_stream_t stream);

/* bacs_proto_accumulate in the exact mode over the GLOBAL view of a data-parallel batch: this rank's images are
 * rows of the D x N_t view of one process fed every rank's images in rank order (rank 0's first).  view_pre[t]
 * (int64, device) counts task t's masked pixels in the images of the ranks below this one, view_n[t] over all ranks;
 * image b's entry of channel c lands in row (D*(view_pre[t] + pre_bt) + c*n_bt) / view_n[t].  Summing the ranks'
 * sums gives the exact sums of the concatenated batch.  counts stay LOCAL (the exchange of the sums adds them up).
 * The view's values are read on the device and must satisfy view_pre[t] + sum_b n_bt[b][t] <= view_n[t], or
 * view_n[t] < 0: an invalid view (a peer time-out of bacs_peer_count_exchange), for which task t adds nothing and
 * counts[t] = -inf, so the running-mean update of bacs_proto_update / bacs_peer_allreduce skips it.
 * NULL view_pre and view_n: the local view, i.e. exactly bacs_proto_accumulate.  BACS_ERR_INVALID before any launch
 * when only one of the two is given, T is not in [1, BACS_MAX_TASKS] or a view comes with mode != 0. */
int bacs_proto_accumulate_view(const void* features, int dtype, int B, int D, int h, int w,
                               const int8_t* task, const int32_t* rank, const int32_t* n_bt, int T,
                               int mode, const int64_t* view_pre, const int64_t* view_n, double* sums,
                               double* counts, void* workspace, size_t workspace_bytes, bacs_stream_t stream);

/* Count exchange without peer memory: totals[t] = sum_b n_bt[b][t] (int64[T]), the payload of an all-gather into a
 * [world][T] table; bacs_proto_count_view turns that table into rank `rank`'s view (sums in rank order). */
int bacs_proto_task_totals(const int32_t* n_bt, int B, int T, int64_t* totals, bacs_stream_t stream);
int bacs_proto_count_view(const int64_t* table, int world, int rank, int T, int64_t* view_pre, int64_t* view_n,
                          bacs_stream_t stream);

/* Running-mean update proto[g] = (S[g] + cnt[g]*proto[g]) / (cnt[g] + N[g]); cnt[g] += N[g]
 * for rows with N[g] > 0 (prototypes.py:158-163), fp32 arithmetic like torch's.
 * count_is_int64: the reference keeps int64 counts at task 0 and float32 afterwards (Q3).
 * ready (int32[1]) = all counts non-zero after the update (prototypes.py:31-40). */
int bacs_proto_update(float* proto, void* count, int count_is_int64, const double* sums,
                      const double* counts, int T, int D, int32_t* ready, bacs_stream_t stream);

/* ---------------------------------------------------------------------------------
 * Seen / unseen detector heads (networks/bg_detector.py:17-40, 100-165)
 * --------------------------------------------------------------------------------- */

/* z[b,t,q] = bias[t] + sum_c weight[t,c] * |sigmoid(f[b,c,q]) - sigmoid(proto[t,c])| at
 * feature resolution.  The x16 bilinear up-sample (align_corners=True), sigmoid and
 * max over heads are evaluated inside the consumers, so [B,T,H,W] never exists. */
int bacs_seen_logits(const void* features, int dtype, int B, int D, int h, int w,
                     const float* proto, const float* weight, const float* bias, int T,
                     float* z, bacs_stream_t stream);

/* The same with the T heads given as they live in the model: HOST arrays of T device pointers (weight_rows_host[t] ->
 * fp32[D], bias_host[t] -> fp32[1]; the nn.Conv2d parameters of bg_detector.py:17-40), so no gather launch precedes
 * the kernel.  zero_out (optional, fp32[B,h,w]) is cleared by the same launch: it is the focal-gradient accumulator
 * `gz` of the bacs_pixel_loss call that follows. */
int bacs_seen_logits_heads(const void* features, int dtype, int B, int D, int h, int w,
                           const float* proto, const float* const* weight_rows_host,
                           const float* const* bias_host, int T, float* z, float* zero_out,
                           bacs_stream_t stream);

/* Any number of heads 1 <= T <= BACS_MAX_TASKS (continual runs longer than 32 tasks).  The heads come as host arrays
 * of device pointers as in bacs_seen_logits_heads, or, when weight_rows_host is NULL, stacked as weight fp32[T,D] and
 * bias fp32[T] as in bacs_seen_logits.  zero_out as in bacs_seen_logits_heads (may be NULL).  One launch: a grid
 * dimension over chunks of 32 heads, each evaluated with the T = 32 plan of bacs_seen_logits; the chunks after the
 * first read the features mostly from L2.  At T <= 32 the result equals bacs_seen_logits' bit for bit when both
 * launches split the channels over the same cluster size. */
int bacs_seen_logits_many(const void* features, int dtype, int B, int D, int h, int w,
                          const float* proto, const float* weight, const float* bias,
                          const float* const* weight_rows_host, const float* const* bias_host, int T,
                          float* z, float* zero_out, bacs_stream_t stream);

/* Materialised seen logits of the reference for callers that need the full-res map
 * (get_seen_map_task / get_seen_probs, bg_detector.py:100-165): out[b,t,Y,X] =
 * (apply_sigmoid ? sigmoid : id)(bilinear_ac_true(z[b,t])) with H = h*scale. */
int bacs_seen_upsample(const float* z, int B, int T, int h, int w, int scale, int apply_sigmoid,
                       float* out, bacs_stream_t stream);

/* Backward of one head (focal path, base_loss.py:255-272): given gz = dL/dz[b,q] for the
 * head, accumulate dweight[D], dbias[1] (fp32, OVERWRITTEN) and, when dfeatures != NULL
 * (first task: stop_gradients False), dfeatures[B,D,h,w] (dtype, OVERWRITTEN).
 * scale_dev: optional device float[1] multiplied into every gradient (normaliser that
 * is only known on the device), NULL = 1. */
int bacs_seen_head_backward(const void* features, int dtype, int B, int D, int h, int w,
                            const float* proto_t, const float* weight_t, const float* gz,
                            const float* scale_dev, float* dweight, float* dbias,
                            void* dfeatures, bacs_stream_t stream);

/* Device-side normaliser of the focal term (base_loss.py:221-222,242-250,260-262):
 *   scale = weight * [ready] * [#background pixels > 0] / #kept pixels, read from the
 *   accumulators of bacs_pixel_loss (acc) and bacs_proto_update (ready, may be NULL).
 *   scale_out float[1] (for bacs_seen_head_backward); out2 double[2] = {scale,
 *   scale * acc[BACS_ACC_FOCAL]} (for bacs_combine_scalars).  Either may be NULL. */
int bacs_focal_scale(const double* acc, const int32_t* ready, float weight, float* scale_out,
                     double* out2, bacs_stream_t stream);
/* The same plus the loss scalar of the fused per-pixel Function in one launch:
 *   loss_out float[1] = main_coef * acc[BACS_ACC_LOSS] / (main_over_wsum ? acc[BACS_ACC_WSUM] : 1)
 *                       + scale * acc[BACS_ACC_FOCAL]. */
int bacs_focal_scale_loss(const double* acc, const int32_t* ready, float weight, float main_coef,
                          int main_over_wsum, float* scale_out, float* loss_out, bacs_stream_t stream);

/* ---------------------------------------------------------------------------------
 * The fused per-pixel kernel: softmax statistics read ONCE per pixel, then
 *   mode BACS_PIX_WEIGHTED_CE : background-aware unbiased CE (training/loss_utils.py:542-585)
 *                               [+ seen-detector focal loss of one head, base_loss.py:255-272]
 *                               [+ teacher-distill pixel mask, bacs_loss.py:282-285]
 *   mode BACS_PIX_CE          : plain / class-weighted CE (base_loss.py:237-240)
 *                               [+ focal loss of one head on the first task]
 *   mode BACS_PIX_UNBIASED_CE : MiB unbiased CE (training/loss_utils.py:492-520)
 *   mode BACS_PIX_SCORE       : per-image importance  -(w_y nll).mean (bacs_loss.py:183-189)
 * plus arg-max (bacs_loss.py:255) and the gradient w.r.t. the logits in the same pass.
 * --------------------------------------------------------------------------------- */
enum bacs_pixel_mode {
  BACS_PIX_WEIGHTED_CE = 0,
  BACS_PIX_CE = 1,
  BACS_PIX_UNBIASED_CE = 2,
  BACS_PIX_SCORE = 3
};

/* slots of the fp64 accumulator vector produced by bacs_pixel_loss */
enum bacs_pixel_acc {
  BACS_ACC_LOSS = 0,        /* sum of per-pixel CE terms (un-normalised) */
  BACS_ACC_WSUM = 1,        /* sum of class weights over valid pixels (CE normaliser) */
  BACS_ACC_FOCAL = 2,       /* sum of focal terms over kept pixels */
  BACS_ACC_KEPT = 3,        /* # pixels with label != ignore */
  BACS_ACC_BG = 4,          /* # pixels with label == 0 */
  BACS_ACC_INVALID = 5,     /* # labels outside [0,K) that are not ignore (treated as ignore) */
  BACS_ACC_DISTILL_PIX = 6, /* # pixels in the teacher-distill mask */
  BACS_ACC_VALID = 7,       /* # pixels with a valid class label */
  BACS_NACC = 8
};

typedef struct bacs_pixel_args {
  const void* logits;     /* [B,K,H,W] */
  const int64_t* labels;  /* [B,H,W] */
  void* dlogits;          /* [B,K,H,W] same dtype as logits, or NULL (no gradient) */
  int64_t* preds;         /* [B,H,W] arg-max (ties -> lowest channel), or NULL */
  const float* z;         /* [B,T,h,w] low-res seen logits, or NULL */
  const float* seen_max;  /* [B,H,W] max_t seen probability already at full resolution, or NULL;
                             when given it replaces sigmoid(max_t upsample(z)) in the CE
                             modulation and the distill mask (stand-alone WeightedCrossEntropy
                             API, training/loss_utils.py:586-588) */
  uint8_t* distill_mask;  /* [B,H,W] out: (label==0) & (max_t seen > lkd_threshold), or NULL */
  float* gz;              /* [B,h,w] out: d(focal sum)/dz of head focal_head, atomically
                             accumulated (caller zeroes), or NULL = no focal term */
  const float* class_w;   /* [K] class weights (CE / SCORE modes) or NULL = ones */
  const int64_t* hist;    /* [257] label histogram: needed when class_w != NULL or mode is
                             CE/UNBIASED_CE and dlogits != NULL (gradient normaliser); such a
                             gradient request needs K <= 256, since the histogram's last bin
                             counts every label >= 256 together */
  double* acc;            /* [BACS_NACC] OVERWRITTEN with the reduced accumulators */
  double* score;          /* [B] per-image score (SCORE mode), or NULL */
  int32_t B, K, H, W, T, h, w;
  int32_t dtype, mode;
  int32_t old_cl, ukd;    /* WEIGHTED_CE / UNBIASED_CE */
  int32_t focal_head;     /* head index in z used by the focal term */
  int32_t ignore_index;
  int32_t seen_scale;     /* H == h * seen_scale (nn.Upsample(scale_factor=16)) */
  float gamma, threshold; /* WEIGHTED_CE focal modulation (1 - s)^gamma, s>thr -> 1 */
  float focal_gamma;
  float focal_alpha;      /* < 0 = no alpha weighting */
  float lkd_threshold;
  float grad_scale;       /* static multiplier folded into dlogits (e.g. beta) */
  /* Optional epilogue evaluated by the reduction launch (saves two single-thread launches per step):
   *   focal_scale_out[0] = focal_weight * [ready] * [#background > 0] / #kept      (as bacs_focal_scale)
   *   loss_out[0] = loss_coef * acc[LOSS] / (loss_over_wsum ? acc[WSUM] : 1) + focal_scale * acc[FOCAL]
   * Both pointers NULL = off. */
  const int32_t* ready;   /* device flag of bacs_proto_update, or NULL = ready */
  float* focal_scale_out; /* float[1] or NULL */
  float* loss_out;        /* float[1] or NULL */
  float focal_weight;
  float loss_coef;
  int32_t loss_over_wsum;
} bacs_pixel_args;

size_t bacs_pixel_workspace_bytes(const bacs_pixel_args* args_host);
/* Which kernel serves these arguments: 0 = generic shared-memory tiles (any K, ragged shapes),
 * 1 = register-resident tiles (K <= 24), 2 = the training-step specialisation (WEIGHTED_CE on
 * 512-pixel row tiles), 4 = two streaming passes (K >= 64: fp32 logits, per-image scores, K > 152),
 * 5 = one pass with the channel column of a pixel pair in registers (64 <= K <= 152, 16-bit logits,
 * H*W a multiple of 256), -1 = no plan.  Introspection only (tests, bench labels). */
int bacs_pixel_kernel_variant(const bacs_pixel_args* args_host);
int bacs_pixel_loss(const bacs_pixel_args* args_host, void* workspace, size_t workspace_bytes,
                    bacs_stream_t stream);

/* The same loss evaluated straight from the network's LOW-RES logits (SURVEY 8f-1): replaces
 *   logits = F.interpolate(sem_logits, size=(H,W), mode="bilinear", align_corners=False)
 * of networks/deeplab_v3.py:154-160 (forward AND its autograd backward) together with the loss it feeds, so no
 * [B,K,H,W] logit or gradient tensor exists.  Arguments as bacs_pixel_loss except
 *   args->logits  = sem_logits [B,K,lh,lw]   (model(x, return_sem_logits=True), deeplab_v3.py:155-156)
 *   args->dlogits = d loss / d sem_logits [B,K,lh,lw], same dtype (or NULL)
 *   args->H, W    = label resolution: W == s * lw with s = 8 or 16 and H a multiple of lh, or, for an input of any
 *                   size, lh == ceil(H / s) and lw == ceil(W / s) with s = 8 or 16 (the network's output stride);
 *                   lw <= 256, K <= 255.  The seen logits args->z (focal term, WEIGHTED_CE's seen probabilities)
 *                   need the first form, i.e. inputs that are multiples of 16 at seen_scale 16; args->seen_max
 *                   works with both.  An unsupported geometry returns BACS_ERR_UNSUPPORTED (workspace size 0).
 * Workspace: bacs_pixel_lowres_workspace_bytes.  Asynchronous on `stream`; gradients are accumulated with fp32
 * atomics (summation order is not fixed: results agree to fp32 rounding, not bit for bit, between runs). */
size_t bacs_pixel_lowres_workspace_bytes(const bacs_pixel_args* args_host, int32_t lh, int32_t lw);
int bacs_pixel_loss_lowres(const bacs_pixel_args* args_host, int32_t lh, int32_t lw, void* workspace,
                           size_t workspace_bytes, bacs_stream_t stream);

/* ---------------------------------------------------------------------------------
 * Pseudo-labelled background (loss/bacs_loss.py:205-210):
 *   pseudo = argmax_c teacher[:, c];  labels[labels == 0] = pseudo[labels == 0]
 * in place on labels int64 [B,H,W]: where a label is 0 it becomes the teacher's arg-max (ties -> lowest channel);
 * every other value (255, other classes, negative or out-of-range values) keeps its bits.  K_t, the teacher's channel
 * count, may differ from the student's; dtype is the teacher's (fp32, bf16, fp16).  Asynchronous on `stream`, no
 * workspace, no host synchronisation (graph-capturable).  Null pointers or B, K_t, H, W <= 0 give BACS_ERR_INVALID.
 *
 * bacs_pseudo_label: full-resolution teacher logits [B,K_t,H,W] (NCHW), any K_t >= 1.
 * bacs_pseudo_label_lowres: the teacher's low-res sem_logits [B,K_t,lh,lw]; the bilinear align_corners=False
 *   up-sample to H x W is evaluated inside the arg-max, and the result equals bit for bit the preds of
 *   bacs_pixel_loss_lowres for the same sem_logits.  Geometry: what bacs_pixel_loss_lowres accepts without z (K = K_t);
 *   anything else returns BACS_ERR_UNSUPPORTED and leaves the labels untouched.
 * --------------------------------------------------------------------------------- */
int bacs_pseudo_label(const void* teacher, int32_t dtype, int32_t B, int32_t K_t, int32_t H, int32_t W,
                      int64_t* labels, bacs_stream_t stream);
int bacs_pseudo_label_lowres(const void* sem_logits, int32_t dtype, int32_t B, int32_t K_t, int32_t lh, int32_t lw,
                             int32_t H, int32_t W, int64_t* labels, bacs_stream_t stream);

/* ---------------------------------------------------------------------------------
 * Teacher distillation on the last attention map (loss/bacs_loss.py:258-294):
 *   L = lkd * mean_{b,a,y} sqrt( sum_x ( m * (U(old)^2 - U(new)^2) )^2 ),
 *   U = bilinear up-sample to HxW, align_corners=False; gradient to `new` only.
 * mask u8[B,H,W] (from bacs_pixel_loss) or NULL = all ones.
 * loss_sum fp64[1] OVERWRITTEN with sum over rows of the row norms (caller scales by
 * lkd / (B*A*H)); loss_scaled fp32[1] OVERWRITTEN with grad_coef * that sum (the loss term itself when
 * grad_coef = lkd / (B*A*H)), or NULL; dnew (dtype, [B,A,h,w]) OVERWRITTEN with grad_coef * d(sum)/dnew, or NULL.
 * Two kernels serve the call: the GEMM form on the 5th-generation tensor cores (csrc/distill_tc.cu: tcgen05.mma,
 * TMEM operands, split-tf32; attention rows of 32 / 64 / 128 bytes, w <= 32, 16-byte aligned pointers) and the
 * generic packed-fp32 kernel (csrc/distill.cu) for every other shape.  bacs_distill_kernel_variant tells which one
 * a shape gets (1 = tensor cores, 0 = FMA kernel); bacs_distill_set_mode(0 auto | 1 FMA only | 2 tensor cores or
 * BACS_ERR_UNSUPPORTED) is a process-wide switch for A/B measurements and tests.
 * --------------------------------------------------------------------------------- */
size_t bacs_distill_workspace_bytes(int B, int A, int h, int w, int H, int W);
int bacs_distill_set_mode(int mode);
int bacs_distill_kernel_variant(int dtype, int B, int A, int h, int w, int H, int W);
int bacs_teacher_distill(const void* old_att, const void* new_att, int dtype, int B, int A,
                         int h, int w, const uint8_t* mask, int H, int W, float grad_coef,
                         double* loss_sum, float* loss_scaled, void* dnew, void* workspace,
                         size_t workspace_bytes, bacs_stream_t stream);
/* The same with loss_scaled[0] = addend[0] + grad_coef * sum (addend: device fp32[1], e.g. the loss terms that precede
 * the distillation term in BACSLoss.compute_loss, bacs_loss.py:250-253): the step's loss scalar without an add launch. */
int bacs_teacher_distill_add(const void* old_att, const void* new_att, int dtype, int B, int A,
                             int h, int w, const uint8_t* mask, int H, int W, float grad_coef,
                             double* loss_sum, float* loss_scaled, const float* addend, void* dnew,
                             void* workspace, size_t workspace_bytes, bacs_stream_t stream);

/* ---------------------------------------------------------------------------------
 * Dark-experience-replay logit MSE with transplant (loss/bacs_loss.py:387-431)
 *   memory logits: fp32 (truncated toward zero in-kernel when `truncate`, reproducing
 *   preprocess_batch's .long(), base_loss.py:274-282) or int64 (memory_is_int64).
 *   cut int32[Br]: first channel of sample j replaced by the live logits (host computes
 *   it with the reference's unique/inverse quirk, Q5); ignore_rep_bg replaces channel 0.
 * loss_sum fp64[1] OVERWRITTEN with sum of squared differences; dsem (dtype) OVERWRITTEN
 * with grad_coef * 2 (s - m), or NULL.
 * --------------------------------------------------------------------------------- */
int bacs_der_mse(const void* sem_logits, int dtype, const void* memory_logits, int memory_is_int64,
                 int truncate, const int32_t* cut, int ignore_rep_bg, int Br, int K, int hw,
                 float grad_coef, double* loss_sum, void* dsem, void* workspace,
                 size_t workspace_bytes, bacs_stream_t stream);
size_t bacs_der_workspace_bytes(int Br, int K, int hw);
/* cut[j] from the stored class counts n_classes int64[Br] (values < 1024), on the device,
 * reproducing `for i, n in enumerate(unique(n_classes)): j = inverse[i]` (Q5). */
int bacs_der_cut(const int64_t* n_classes, int Br, int K, int32_t* cut, bacs_stream_t stream);

/* ---------------------------------------------------------------------------------
 * MiB unbiased knowledge distillation (training/loss_utils.py:447-489).  Instantiated on every
 * loss object (base_loss.py:78) but called only by the MiB / SDR losses.
 *   logits [B,K,H,W], old_logits [B,K_old,H,W] (same dtype), mask u8[B,H,W] or NULL.
 *   loss_sum fp64[1] OVERWRITTEN with sum_p mask * per_p (caller: loss = -loss_sum / (B*H*W));
 *   dlogits (dtype) OVERWRITTEN with grad_coef * d(-sum)/dlogits, or NULL.
 * --------------------------------------------------------------------------------- */
size_t bacs_unbiased_kd_workspace_bytes(int64_t npix);
int bacs_unbiased_kd(const void* logits, const void* old_logits, int dtype, int B, int K, int K_old,
                     int H, int W, float alpha, const uint8_t* mask, float grad_coef,
                     double* loss_sum, void* dlogits, void* workspace, size_t workspace_bytes,
                     bacs_stream_t stream);

/* ---------------------------------------------------------------------------------
 * Confusion matrix (training/metrics.py:38-88 over torchmetrics 0.6.0 ConfusionMatrix)
 * --------------------------------------------------------------------------------- */
/* confmat[t*K + p] += 1 for pixels with 0 <= t < K (rows = target).  preds are int64
 * (preds_is_float = 0) or fp32 truncated like .int() (metrics.py:45-46).  Predictions
 * outside [0,K) on a kept pixel are counted in oob[0] (torch.bincount would have
 * enlarged / raised); confmat int64[K*K] is accumulated in place. */
int bacs_confmat_accumulate(const void* preds, int preds_is_float, const int64_t* target,
                            int64_t n, int K, int64_t* confmat, int64_t* oob,
                            bacs_stream_t stream);
/* per-class metrics from the matrix with the reference's naming (metrics.py:52-88):
 * out fp32[6,K] = iou, accuracy, precision, recall, specificity, (row 5: miou broadcast) */
int bacs_confmat_metrics(const int64_t* confmat, int K, float* out, bacs_stream_t stream);

/* ---------------------------------------------------------------------------------
 * Small device-side helpers so the step stays free of host synchronisation
 * --------------------------------------------------------------------------------- */
/* ---------------------------------------------------------------------------------
 * OPTIONAL per-class prototype family (SURVEY 8f-4, BASELINE.json north_star): squared distance of every pixel's
 * feature vector to every class prototype on the tcgen05 tensor cores,
 *   dist2[b,k,y,x] = max(|f|^2 + |c_k|^2 - 2 <f, c_k>, 0),   nearest[b,y,x] = argmin_k (ties -> lowest class).
 * Not reference arithmetic (the reference's heads are a weighted L1 of sigmoids, networks/bg_detector.py:17-40; SDR,
 * loss/sdr.py:120-200, only ever touches a pixel's own class): the building block for nearest-class-prototype maps
 * at ADE20K sizes (150 x 512 prototypes).  features [B,D,h,w] and protos [Kc,D] are bf16 (dtype = BACS_BF16), fp32
 * accumulation; h*w and D multiples of 8, D <= 512, Kc <= 256 and the prototypes (padded to a multiple of 32 classes)
 * resident in one SM's shared memory next to 32 KB of staging (<= 224 KB; 150 x 512 fits); BACS_ERR_UNSUPPORTED
 * otherwise.  One hand-written kernel (csrc/class_distance.cu): TMA -> tensor memory (A) / shared memory (B) ->
 * tcgen05.mma -> norms, clamp and arg-min in the epilogue.  The workspace is not used (size query kept for callers).
 * nearest may be NULL.
 * --------------------------------------------------------------------------------- */
size_t bacs_class_distance_workspace_bytes(int32_t B, int32_t Kc, int32_t D, int32_t h, int32_t w);
int bacs_class_distance(const void* features, int dtype, int32_t B, int32_t D, int32_t h, int32_t w, const void* protos,
                        int32_t Kc, float* dist2, int64_t* nearest, void* workspace, size_t workspace_bytes,
                        bacs_stream_t stream);

/* Per-class feature sums of the same family (SDR's per-class prototypes, loss/sdr.py:120-159; the segmented reduction
 * of bacs_proto_accumulate with one group per CLASS instead of per task): sums[k][c] = sum over the low-res pixels of
 * class k of features[b][c][pixel], fp64 [K, D], OVERWRITTEN.  labels_down int64 [B,h,w] holds class ids (what
 * bacs_label_downsample_task returns as labels_down); ids outside [0, K) -- ignore-255 -- are skipped.  The per-class
 * pixel counts are bacs_label_hist of the same labels.  workspace >= bacs_class_sums_workspace_bytes. */
size_t bacs_class_sums_workspace_bytes(int32_t B, int32_t D, int32_t K);
int bacs_class_sums(const void* features, int dtype, int32_t B, int32_t D, int32_t h, int32_t w,
                    const int64_t* labels_down, int32_t K, double* sums, void* workspace,
                    size_t workspace_bytes, bacs_stream_t stream);

/* Minibatch gather of the HBM-resident replay store (SURVEY 8f-2): dst[i] = src[idx[i]] for rows of row_bytes bytes.
 * Replaces the fancy-index read of the reference's memmapped buffer fields in Buffer.get_data
 * (training/buffer.py:371-381) and BaseMemMapDataset.__getitem__ (dataset/base_segmentation_dataset.py:89-97) plus
 * the host->device copy of the sampled batch.  idx: device int64[n_idx]; an index outside [0, n_rows) gives a zero
 * row.  16-byte vector path when row_bytes, src and dst are 16-byte aligned. */
int bacs_gather_rows(const void* src, int64_t n_rows, int64_t row_bytes, const int64_t* idx, int64_t n_idx, void* dst,
                     bacs_stream_t stream);

/* In-place x *= *g for a gradient tensor when the upstream gradient is not 1; the kernel
 * exits immediately (uniformly) when *g == 1. */
int bacs_scale_inplace(void* x, int dtype, int64_t n, const float* g_dev, bacs_stream_t stream);
/* The same for up to 8 tensors in one launch (x[i] may be NULL: skipped). */
int bacs_scale_inplace_multi(int n, void* const* x, const int* dtype, const int64_t* numel,
                             const float* g_dev, bacs_stream_t stream);

/* out[0] = sum_i coef[i] * src[i][idx[i]] / (den[i] ? den[i][didx[i]] : 1), n <= 8 terms:
 * assembles the step's loss scalar on the device from the fp64 accumulators.  src/den
 * are HOST arrays of device pointers; idx/didx/coef are host arrays. */
int bacs_combine_scalars(int n, const double* const* src_host, const int* idx_host,
                         const double* const* den_host, const int* didx_host,
                         const float* coef_host, float* out, bacs_stream_t stream);

/* One-shot all-reduce (sum) of the packed fp64 state over NVLink PEER MEMORY, optionally fused with the
 * prototype running-mean update of bacs_proto_update (pass proto = NULL for the plain all-reduce):
 * no counterpart in the reference (each DDP rank keeps its own prototypes, loss/prototypes.py:157-163).
 *   peer_buf_host[r]  : device address, valid on THIS GPU, of rank r's symmetric region of 2*n_max doubles
 *   peer_flag_host[r] : device address of rank r's flag row of >= 16 zero-initialised uint32
 *   step_dev          : device uint32 step counter of this rank (0 at start; the kernel increments it, so
 *                       the call can be replayed from a CUDA graph)
 *   error_dev         : sticky device int32 (or NULL): receives the step number when a peer did not show up
 *                       within the time-out (bacs_peer_set_timeout_ms, default 30 s; the kernel never hangs).
 *                       On a time-out NOTHING is combined: packed, proto, count are left untouched and
 *                       *ready = 0 -- the caller must check error_dev at its next synchronisation point and fail.
 * Every rank must make the same sequence of calls.  packed is summed in rank order: all ranks obtain
 * bit-identical results. */
int bacs_peer_allreduce(double* packed, int n, int n_max, int rank, int world,
                        const uint64_t* peer_buf_host, const uint64_t* peer_flag_host, uint32_t* step_dev,
                        int32_t* error_dev, float* proto, void* count, int count_is_int64, int T, int D,
                        int32_t* ready, bacs_stream_t stream);

/* Count phase of the global prototype view over NVLink PEER MEMORY (one launch, no host synchronisation,
 * graph-capturable): this rank's task totals sum_b n_bt[b][t] are pushed into every peer's count table, and after
 * every peer has published, view_pre / view_n (int64[T], the inputs of bacs_proto_accumulate_view) are summed from
 * the local table in rank order.
 *   peer_table_host[r] : device address of rank r's count table of 2 * world * BACS_MAX_TASKS int64
 *   peer_flag_host[r]  : device address of rank r's count-flag row of >= 16 zero-initialised uint32, apart from
 *                        the flag row of bacs_peer_allreduce
 *   step_dev           : device uint32 step counter of the count phase (its own, not that of the sums)
 *   error_dev          : sticky device int32 (or NULL), as in bacs_peer_allreduce.
 * On a time-out the view is marked invalid (view_pre = 0, view_n = -1) and error_dev receives the count step: the
 * accumulate launch adds nothing and reports -inf counts, so the update after the exchange of the sums leaves this
 * rank's prototypes and counts untouched for the step; the caller must check error_dev and fail.  Every rank must
 * make the same sequence of calls. */
int bacs_peer_count_exchange(const int32_t* n_bt, int B, int T, int rank, int world, const uint64_t* peer_table_host,
                             const uint64_t* peer_flag_host, uint32_t* step_dev, int32_t* error_dev,
                             int64_t* view_pre, int64_t* view_n, bacs_stream_t stream);

/* Wall-clock bound (milliseconds, > 0) of the peer wait of bacs_peer_allreduce; process-wide. */
int bacs_peer_set_timeout_ms(int64_t ms);

/* Pack / unpack the per-step cross-rank state into ONE fp64 buffer for a single
 * all-reduce: [T*D prototype sums | T counts | K*K confusion matrix (optional)]. */
int bacs_pack_state(const double* sums, const double* counts, int T, int D,
                    const int64_t* confmat, int K, double* packed, bacs_stream_t stream);
int bacs_unpack_state(const double* packed, int T, int D, double* sums, double* counts,
                      int64_t* confmat, int K, bacs_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* BACS_B200_H_ */
