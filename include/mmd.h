/*
 * mmd.h — C ABI of libmmd_b200.so: the sm_100a kernels behind the MM-DistillNet distillation hot path.
 *
 * The reference (robot-learning-freiburg/MM-DistillNet) is pure PyTorch and has no FFI for this path; the
 * "interface each entry point replaces" is therefore the reference's Python call site:
 *
 *   mmd_mta_fwd / mmd_mta_bwd      replace  MTALoss.forward / .mtaloss / .at and their autograd
 *                                           (src/loss/MTALoss.py:15-34, :36-74, :76-77)
 *   mmd_focal_fwd / mmd_focal_bwd  replace  YetAnotherFocalLoss.forward and its autograd (src/loss/YetAnotherFocalLoss.py:27-190)
 *   mmd_pseudo_labels              replaces logits_to_ground_truth / EfficientDet_post_processing per teacher
 *                                           (src/utils/utils.py:144-231, :234-324) and the cross-teacher integration + nms of
 *                                           the step wrappers (src/optimization/train_methods.py:186-250, :343-411)
 *   mmd_adam_step                  replaces torch.optim.Adam / AdamW .step() over the student's parameters
 *                                           (constructed at src/optimization/train_methods.py:825-842, stepped at
 *                                            src/optimization/traditional.py:190)
 *   mmd_bifpn_run                  replaces nn.Sequential(*[BiFPN(...)]) forward and its autograd
 *                                           (src/YetAnotherEfficientDet.py:639-644, :668; one cell :320-392;
 *                                            SeparableConvBlock.forward :182-192; same-pad conv / pool
 *                                            src/YetAnotherEfficientNet.py:51-65, :90-104; swish :126-137)
 *
 * Conventions: plain pointers and sizes only (no torch types).  Every pointer is a DEVICE pointer borrowed for
 * the duration of the call; nothing is allocated or freed inside; all work is enqueued asynchronously on the
 * caller's stream (a cudaStream_t passed as void*) and never synchronises the host, so calls are CUDA-graph
 * capture safe.  Return value 0 = OK, otherwise a cudaError_t (or a negative MMD_E* argument error); the message
 * is available from the thread-local mmd_last_error().  No exceptions cross the ABI.
 *
 * Layout: activations are NHWC ([B][H][W][C], i.e. torch channels_last of a logical [B,C,H,W] tensor) unless a
 * call says otherwise; parameters are the reference's own fp32 tensors in their native PyTorch layouts
 * (depthwise [C,1,3,3], pointwise [Cout,Cin,1,1], BatchNorm vectors [C]) — the kernels fold / transpose on load,
 * so no packed copies can go stale.
 */
#ifndef MMD_H
#define MMD_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MMD_VERSION 111

typedef void* mmd_stream_t; /* cudaStream_t */

enum { MMD_F32 = 0, MMD_BF16 = 1 };               /* storage type of activations (arithmetic is fp32) */
enum { MMD_NHWC = 0, MMD_NCHW = 1 };              /* MTA accepts both; BiFPN is NHWC only */
enum { MMD_E_ARG = -1, MMD_E_UNSUPPORTED = -2 };

int mmd_version(void);
const char* mmd_last_error(void);
/* number of kernels this library has launched in the calling process (all threads); for bench accounting */
unsigned long long mmd_launch_count(void);

/* ------------------------------------------------------------------------------------------------------------
 * MTA loss (src/loss/MTALoss.py).  One call handles every pyramid level and every teacher.
 *   a = mean_c f^p ; a^ = a / max(||a||_2, 1e-12) ; teachers: product of a^_k, L1-renormalised when n_teachers>1
 *   loss[l] = sum_b sum_i t (log t - s) / B  with s = softmax(a^_s/T), t = softmax(a^_t/T)   (reference quirk:
 *   probabilities, not log-probabilities, are the kl_div input — reproduced as is).
 * ---------------------------------------------------------------------------------------------------------- */
#define MMD_STATS_REPLICAS 1
#define MMD_MTA_MAX_LEVELS 8
#define MMD_MTA_MAX_TEACHERS 4

typedef struct {
  int32_t n_levels, n_teachers, B, C;
  int32_t dtype;  /* MMD_F32 / MMD_BF16 : element type of fs / ft / grad_fs */
  int32_t layout; /* MMD_NHWC / MMD_NCHW */
  float T, p;
  int32_t separate; /* 0: ONE loss call against the product of all n_teachers (MTALoss.py:20-34).                 */
                    /* 1: n_teachers independent single-teacher calls that share the student (what the step       */
                    /*    wrappers do, train_methods.py:351-358: criterion_kd(features_s, features_t) per teacher) */
                    /*    in one set of launches: the student maps are pooled once; loss / loss_b / ga_ws hold    */
                    /*    n_teachers consecutive results ([call][level], [call][level][B], [call][B*sum HW]) and  */
                    /*    mmd_mta_bwd takes grad_loss[call][level] and writes the SUM of the calls' gradients.    */
  int32_t pad_;
  int32_t H[MMD_MTA_MAX_LEVELS], W[MMD_MTA_MAX_LEVELS];
  const void* fs[MMD_MTA_MAX_LEVELS];                       /* student features, one per level            */
  const void* ft[MMD_MTA_MAX_TEACHERS][MMD_MTA_MAX_LEVELS]; /* teacher features [teacher][level]          */
  float* att_ws;  /* workspace, (1+n_teachers) * B * sum_l(H*W) floats: channel-pooled maps a              */
  float* ga_ws;   /* workspace, B * sum_l(H*W) floats: d loss[l] / d a_s (per unit upstream grad); may be  */
                  /* NULL for a forward that will never be differentiated                                  */
  float* loss_b;  /* workspace, n_levels * B floats: per-sample loss terms                                 */
  float* loss;    /* out, n_levels floats                                                                  */
} MmdMtaArgs;

int mmd_mta_fwd(const MmdMtaArgs* a, mmd_stream_t stream);
/* grad_fs[l] = grad_loss[l] * (p/C) * fs[l]^(p-1) * ga_ws  (same dtype/layout as fs); needs ga_ws from the fwd */
int mmd_mta_bwd(const MmdMtaArgs* a, const float* grad_loss, void* const* grad_fs, mmd_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Detection loss (src/loss/YetAnotherFocalLoss.py:27-190), every sample of the batch in one launch.
 *   per sample b: IoU of every anchor against the sample's boxes (calc_iou :6-20, same operation order in fp32, so the
 *   0.4 / 0.5 decisions are the reference's); max-IoU < 0.4 negative, >= 0.5 positive of the arg-max box's class (first
 *   maximum wins), otherwise ignored; classification scores clamped to [1e-4, 1 - 1e-4]; focal BCE (alpha 0.25, gamma 2)
 *   summed / max(#positives, 1); smooth-L1 (beta 1/9) of the positives' (dy, dx, dh, dw) against the EfficientDet box
 *   encoding, mean over #positives * 4; loss[0] = mean_b regression, loss[1] = mean_b classification.
 *   A sample whose rows are all padding is the reference's "no annotation" branch (all anchors negative, undivided sum).
 *   No valid box in ANY sample: both losses are zeros that do not depend on the predictions (:61-62, :181-188) and every
 *   gradient is zero -- decided on the device (acc[b][3] = valid rows of sample b), so `boxes` may come straight from
 *   mmd_pseudo_labels.  A caller that knows M == 0 on the host simply does not call.
 * ---------------------------------------------------------------------------------------------------------- */
#define MMD_FOCAL_MAX_BOXES 2048
typedef struct {
  int32_t B, N, K, M;      /* samples, anchors, classes, (padded) boxes per sample: 1 <= M <= MMD_FOCAL_MAX_BOXES       */
  int32_t dtype, pad_;     /* MMD_F32 / MMD_BF16: element type of cls / reg and of their gradients                      */
  float alpha, gamma;      /* 0.25, 2.0 in the reference (:44-45); gamma must be 2                                       */
  const void* cls;         /* [B][N][K] sigmoid scores                                                                   */
  const void* reg;         /* [B][N][4] predicted (dy, dx, dh, dw)                                                       */
  const float* anchors;    /* [N][4] (y1, x1, y2, x2), fp32                                                              */
  const float* boxes;      /* [B][M][5] (x1, y1, x2, y2, class), fp32; class == -1 marks a padding row                   */
  double* acc;             /* workspace [B][4]: classification sum, regression sum, #positives, #valid boxes.  Zero on   */
                           /* entry of mmd_focal_fwd; read again by mmd_focal_bwd                                        */
  int32_t* assign;         /* optional out [B][N]: -2 ignored, -1 negative, m >= 0 positive of the sample's m-th valid box */
  float* loss;             /* out [2]: regression_loss, classification_loss                                              */
} MmdFocalArgs;

int mmd_focal_fwd(const MmdFocalArgs* a, mmd_stream_t stream);
/* grad_cls [B][N][K], grad_reg [B][N][4] (dtype of the inputs; every element is written) from the upstream gradients of
 * loss[0] / loss[1] (device scalars; NULL = 0).  Needs `acc` as mmd_focal_fwd left it. */
int mmd_focal_bwd(const MmdFocalArgs* a, const float* grad_reg_loss, const float* grad_cls_loss, void* grad_cls, void* grad_reg,
                  mmd_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Pseudo-label generation (SURVEY.md 8 f3): the teachers' detections become the student's annotations without leaving
 * the device.  Per teacher t and sample b, as EfficientDet_post_processing (src/utils/utils.py:144-231) does:
 *   score = max_k cls[b][n][k] (first maximum = class), kept when score > conf_threshold (:178-179); the class must be a
 *   valid prediction id (:197-204, label_of[class] >= 0); box = YetAnotherEfficientDetBBoxTransform (src/
 *   YetAnotherEfficientDet.py:574-602) of (anchor, regression), clipped by ClipBoxes (:123-141: minima at 0, maxima at
 *   image_size); class-wise NMS = torchvision batched_nms' coordinate trick (class * (max coordinate + 1) added to the
 *   boxes) + greedy NMS in stable descending score order, a kept box suppressing IoU > nms_threshold (:205); rows of an
 *   `ignore` class are dropped AFTER the NMS (:212-215).  Reference quirk kept: the reported score of row j of the
 *   class-filtered list is the score of the j-th over-threshold anchor (:195 indexes the unfiltered list).
 *   logits_to_ground_truth (:291-321): row = [trunc(max(x1,0)), trunc(max(y1,0)), trunc(min(x2,S)), trunc(min(y2,S)),
 *   score, label_of[class]].
 * Then the step wrappers' integration (train_methods.py:360-411): per sample the teachers' rows are concatenated in
 * teacher order, ONE class-agnostic greedy NMS at merge_iou (0.5) over the truncated boxes, the score column dropped:
 *   labels[b][r] = (x1, y1, x2, y2, label) in NMS order, rows >= counts[b] filled with -1 -- exactly the padded
 *   annotation tensor MmdFocalArgs.boxes takes, so the detection loss follows on the same stream with no host round trip.
 * All arithmetic that decides an index (threshold compares, IoU, arg-max, ordering) is fp32 with every operation rounded
 * on its own (no FMA contraction): identical decisions to the fp32 reference.  Launches: 4 for all teachers together.
 * Capacities (the reference has none): at most `cap` over-threshold anchors per (teacher, sample), `max_rows` rows per
 * (teacher, sample) after the NMS, `max_labels` merged rows per sample; anything beyond is dropped in score order and
 * counts[B] (a bit mask: 1 = cap, 2 = max_rows, 4 = max_labels) says so.
 * ---------------------------------------------------------------------------------------------------------- */
#define MMD_PL_MAX_TEACHERS 8
#define MMD_PL_MAX_CAP 8192
#define MMD_PL_MAX_IGNORE 8
typedef struct {
  int32_t B, N, K, T;            /* samples, anchors, classes (<= 255), teachers (<= MMD_PL_MAX_TEACHERS)                     */
  int32_t dtype;                 /* MMD_F32 / MMD_BF16: element type of cls / reg                                             */
  int32_t cap;                   /* <= MMD_PL_MAX_CAP over-threshold anchors per (teacher, sample)                            */
  int32_t max_rows;              /* rows per (teacher, sample) after the class-wise NMS; T * max_rows <= MMD_PL_MAX_CAP       */
  int32_t max_labels;            /* M: rows per sample of `labels` (<= MMD_FOCAL_MAX_BOXES when the loss consumes them)       */
  int32_t raw_rows;              /* 1: teacher_rows = EfficientDet_post_processing's rows (unclipped-to-int boxes, score,     */
                                 /*    class id); 0: logits_to_ground_truth's rows (truncated boxes, score, label)            */
  int32_t n_ignore;
  int32_t ignore[MMD_PL_MAX_IGNORE]; /* prediction ids dropped after the NMS (config 'ignore_labels')                         */
  int32_t merge01;               /* 1: the augmented step (train_methods.py:384-386): when samples 0 and 1 both have rows,    */
                                 /*    sample 1's list = sample 0's rows (all teachers) followed by its own, before the NMS  */
                                 /*    (needs B >= 2 and 2 * T * max_rows <= MMD_PL_MAX_CAP)                                  */
  int32_t pad_;
  float conf_threshold, image_size;
  double nms_threshold, merge_iou;   /* compared as torchvision does: (double)iou > threshold                                 */
  const void* cls[MMD_PL_MAX_TEACHERS]; /* [B][N][K] class probabilities                                                      */
  const void* reg[MMD_PL_MAX_TEACHERS]; /* [B][N][4] (dy, dx, dh, dw)                                                         */
  const float* anchors;          /* [N][4] (y1, x1, y2, x2)                                                                   */
  const int32_t* label_of;       /* [K]: label id of prediction id k, -1 = not a valid prediction id                          */
  void* workspace;               /* mmd_pseudo_workspace_bytes(a) bytes, 16-byte aligned; contents need no initialisation     */
  float* teacher_rows;           /* out [T][B][max_rows][6]                                                                   */
  int32_t* teacher_counts;       /* out [T][B]                                                                                */
  float* labels;                 /* out [B][max_labels][5]                                                                    */
  int32_t* counts;               /* out [B + 1]: merged rows per sample; [B] = overflow bit mask                              */
} MmdPseudoArgs;

size_t mmd_pseudo_workspace_bytes(const MmdPseudoArgs* a);
int mmd_pseudo_labels(const MmdPseudoArgs* a, mmd_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Optimizer step (SURVEY.md 8d, cfg 3): torch.optim.Adam as the reference builds it (train_methods.py:825-833; AdamW :834-842)
 * for every parameter tensor in ONE launch over the flat fp32 gradient buffer of the backward.
 *   t = *step + 1;  m = b1 m + (1 - b1) g;  v = b2 v + (1 - b2) g^2;
 *   p -= lr / (1 - b1^t) * m / (sqrt(v) / sqrt(1 - b2^t) + eps);  then *step = t (a second, 1-thread launch).
 *   weight_decay: g += wd * p (Adam) or p *= 1 - lr * wd first (decoupled_weight_decay = 1, AdamW).
 * Parameter tensors stay the caller's own fp32 tensors (params[i]); grad / exp_avg / exp_avg_sq are flat buffers in which
 * tensor i starts at element offsets[i].  chunks[c] = (tensor, first element inside the tensor, length <= 1024): one CTA each.
 * Everything (tables included) lives on the device; the call is CUDA-graph capture safe.
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct {
  int32_t n_chunks, decoupled_weight_decay;
  int64_t n_elements;            /* sum of the tensors' sizes (profiling only)                                                */
  double lr, beta1, beta2, eps, weight_decay; /* doubles, as the reference's Python scalars: 1 - beta2 is formed in double    */
                                              /* and rounded once (0.001f), not as 1.f - 0.999f                             */
  const int64_t* chunks;         /* device [n_chunks][3]                                                                      */
  const int64_t* offsets;        /* device [n_tensors]                                                                        */
  float* const* params;          /* device [n_tensors] pointers to the fp32 parameter tensors                                 */
  const float* grad;             /* flat gradient                                                                             */
  float* exp_avg;                /* flat first moment (zero before the first step)                                            */
  float* exp_avg_sq;             /* flat second moment (zero before the first step)                                           */
  int64_t* step;                 /* device scalar: number of steps taken so far                                               */
} MmdAdamArgs;

int mmd_adam_step(const MmdAdamArgs* a, mmd_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * BiFPN stack.  The host describes the whole multi-cell forward (or backward) as a flat list of ops over
 * tensors addressed as base[i] + offset, so one op list is built once per shape and replayed with fresh arenas.
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct { int32_t base; int32_t pad_; int64_t off; } MmdRef; /* address = bases[base] + off ; base < 0 : NULL */

typedef struct {
  MmdRef data;      /* NHWC [B][H][W][C], storage dtype                                                        */
  MmdRef bn;        /* NULL: values are final.  Otherwise float[4*C] = scale, shift, mean, invstd of a          */
                    /* train-mode BatchNorm that consumers apply ON LOAD (y = scale*x + shift)                  */
  int32_t H, W, C, pad_;
} MmdTensor;

enum { MMD_IN_SAME = 0, MMD_IN_UP2 = 1, MMD_IN_POOL = 2 };  /* how a node resamples an input (nearest x2 / 3x3 s2 same-pad max) */
enum { MMD_CONS_SAME = 0, MMD_CONS_UP2 = 1, MMD_CONS_POOL = 2 }; /* how a consumer used the tensor whose gradient is gathered */

typedef struct {    /* one gradient source of a tensor (backward is a gather: no atomics on activations) */
  MmdTensor du;     /* the consumer's dL/du (pre-swish fused sum) at the consumer's resolution                  */
  int32_t mode;     /* MMD_CONS_*                                                                               */
  int32_t fw_k, fw_n; /* edge weight = relu(fw[k]) / (sum_j relu(fw[j]) + fw_eps); fw == NULL -> 1             */
  float fw_eps;
  const float* fw;
  MmdRef slot;      /* double[2*C]: sum(G), sum(G*xhat) pushed through this edge by the consumer               */
  MmdRef pidx;      /* uint8 arg-max index per pooled output element (mode POOL)                               */
} MmdCons;

enum {
  MMD_OP_NODE_FWD = 1,  /* fused: resample + BN-on-load + weighted add + swish -> depthwise 3x3 -> pointwise 1x1 (+bias) [-> BN stats] */
  MMD_OP_PROJ_FWD = 2,  /* first-cell 1x1 projection Cin -> C (+bias) [-> BN stats]                                                  */
  MMD_OP_BNAPPLY = 3,   /* out = [pool3x3s2](scale*x + shift): materialise a deferred tensor (P6/P7 synthesis, stack outputs)        */
  MMD_OP_NODE_BWD = 4,  /* backward of NODE_FWD (two kernels: pointwise/BN part, depthwise/fusion part)                              */
  MMD_OP_PROJ_BWD = 5,  /* backward of PROJ_FWD                                                                                      */
  MMD_OP_PULL = 6,      /* dx = gathered gradient of `out` from its consumers (stack inputs, P6/P7 synthesis)                        */
  MMD_OP_SLOT = 7,      /* slot = (sum G, sum G*xhat) for a deferred tensor consumed by a BNAPPLY op                                 */
  MMD_OP_POOLFUSE = 8,  /* bf16 plans: out = w_a * pool3x3s2(bn(in[0])) [+ w_b * bn(in[1])], final values; the pre-pass that turns a  */
                        /* node's pooled input (and its second same-resolution input) into ONE same-resolution operand, so that   */
                        /* every NODE_FWD stages at most two inputs.  pidx[0]: arg-max bytes, save_d: raw value at the arg-max    */
  /* detection heads (Regressor / Classifier, src/YetAnotherEfficientDet.py:445-532): the towers are NODE ops (one input,      */
  /* unweighted), the headers NODE ops with train = 0 on zero-padded weights; these small ops do the rest                     */
  MMD_OP_ACT_FWD = 9,     /* out = swish(in[0])   (in[0] final values): the `alignment` output, :472/:487                      */
  MMD_OP_ACT_BWD = 10,    /* dx  = cons[0].du * swish'(in[0])                                                                  */
  MMD_OP_HEAD_GATHER = 11,/* out[b][head_off + p][k] = act(in[k / C][b][p][k % C]), k < head_K: the header output of one level */
                          /* (n_in = ceil(head_K / C) NHWC tensors padded to C channels) placed into the [B][head_tot][head_K] */
                          /* result, i.e. permute(0,2,3,1) + view + cat(dim=1) (:475-482, :520-530); head_act = 1: sigmoid     */
  MMD_OP_HEAD_SCATTER = 12,/* inverse: in[j] of the forward op = dst j here (`du`, `dd`); cons[0].du = dL/d(result),           */
                          /* out.data = the result itself (sigmoid' = y(1-y)); padding channels are written as zero           */
  MMD_OP_COPY = 13        /* copy_dst[0..copy_n) = copy_src[0..copy_n) (fp32): refresh a zero-padded staging copy of a header's */
                          /* pointwise weight / bias.  Executed by mmd_bifpn_prep (before the packed blocks are rebuilt),      */
                          /* ignored by mmd_bifpn_run                                                                          */
};

typedef struct {
  int32_t kind;
  int32_t train;          /* 1: batch statistics, deferred-BN output, running-stat update (running stats instead: frozen_bn); */
                          /* 0: running stats folded into the 1x1 conv                                                         */
  int32_t n_in;
  int32_t swish;          /* NODE: apply x*sigmoid(x) to the fused sum (BiFPN nodes: 1; bare SeparableConvBlock: 0) */
  MmdTensor in[3];
  int32_t mode[3];        /* MMD_IN_* */
  float fw_eps;
  const float* fw;        /* raw fusion weights [n_in] (fp32 parameter) or NULL for an unweighted sum */
  /* parameters: absolute device pointers to the reference's fp32 tensors */
  const float* dw_w;      /* [C,1,3,3]   (NODE)        */
  const float* pw_w;      /* [C,Cin,1,1]               */
  const float* pw_b;      /* [C]                       */
  const float* bn_w;      /* gamma [C]                 */
  const float* bn_b;      /* beta  [C]                 */
  float* bn_rm;           /* running_mean [C]          */
  float* bn_rv;           /* running_var  [C]          */
  int64_t* bn_nbt;        /* num_batches_tracked       */
  const float* in_bn_w[3];/* gamma / beta of each deferred input's producer (for the fusion-weight gradient) */
  const float* in_bn_b[3];
  int32_t Cin;            /* PROJ: input channels */
  int32_t accumulate_dx;  /* PROJ_BWD / PULL: add into dx instead of overwriting */
  float bn_eps, bn_momentum;
  MmdTensor out;          /* fwd: produced tensor; bwd: the same tensor (its raw values are read again) */
  MmdRef save_d;          /* NODE train: depthwise output kept for the pointwise weight gradient */
  MmdRef pidx[3];         /* NODE / BNAPPLY train: arg-max indices written for pooled inputs */
  MmdRef packed;          /* NODE / PROJ: this op's packed parameter block (written by mmd_bifpn_prep, layout below); */
                          /* NULL: the kernels convert the fp32 parameters themselves (slow path)                 */
  MmdRef stats;           /* double[MMD_STATS_REPLICAS][2*C] accumulators, zero on entry, re-zeroed by the finaliser.  CTAs may  */
                          /* spread their partial sums over the replicas; whoever turns the sums into (scale, shift) adds the    */
                          /* replicas up.  Measured on B200: 16 / 4 / 1 replicas make no difference to the producers, and every  */
                          /* replica costs the consumers of a deferred BatchNorm two more L2 loads per channel: 1 replica.       */
  MmdRef counter;         /* uint32, zero on entry, re-zeroed by the kernel */
  /* backward only */
  int32_t n_cons, pad_;
  MmdCons cons[3];        /* who consumed `out` */
  MmdRef du;              /* NODE_BWD: dL/du written [B][H][W][C] */
  MmdRef dd;              /* NODE_BWD: scratch for dL/d(depthwise output) [B][H][W][C] */
  MmdRef in_slot[3];      /* NODE_BWD: double[2*C] per input edge (zero on entry) */
  MmdRef dx;              /* PROJ_BWD: dL/d(input) [B][H][W][Cin]; PULL: gathered dL/d(out) */
  MmdRef g_dw, g_pw, g_pb, g_bn_w, g_bn_b, g_fw; /* fp32 parameter gradients (zero on entry; accumulated) */
  /* fusion-weight selection for ops that see only part of a node's inputs (NODE_FWD fed by a POOLFUSE, POOLFUSE itself):  */
  int32_t fw_n;           /* number of entries of `fw`; 0: fw has n_in entries and input i uses entry i                      */
  int32_t fw_idx[3];      /* entry of `fw` that weighs input i; -1: the input is already weighted (weight 1)                 */
  /* NODE_BWD of a bf16 node whose forward ran as POOLFUSE + NODE_FWD: what the pre-pass left behind                       */
  MmdRef aux;             /* the pre-weighted operand (pooled input [+ second same-resolution input]), final values         */
  MmdRef praw;            /* raw value of the pooled input at each arg-max (0 where the padding won)                         */
  /* detection heads */
  int32_t head_K, head_tot, head_off, head_act;  /* HEAD_GATHER / HEAD_SCATTER: valid channels, positions per sample of the  */
                                                 /* concatenated result, first position of this level, 1 = sigmoid           */
  const float* copy_src;  /* COPY */
  float* copy_dst;
  int64_t copy_n;
  /* frozen BatchNorm (NODE_FWD / PROJ_FWD / NODE_BWD / PROJ_BWD with train = 1): the layer's nn.BatchNorm2d is in eval()   */
  /* inside a training forward.  mmd_bifpn_prep writes out.bn = (gamma*invstd_r, beta - running_mean*gamma*invstd_r,        */
  /* running_mean, invstd_r), invstd_r = 1/sqrt(running_var + eps), before the forward; the producer accumulates no         */
  /* statistics, finalises nothing and leaves running_mean / running_var / num_batches_tracked untouched; the backward     */
  /* uses A = gamma*invstd_r and no batch-statistics terms (dL/dgamma = sum G*xhat_r, dL/dbeta = sum G as before).         */
  int32_t frozen_bn;
  int32_t pad2_;
} MmdOp;

/* Packed parameter block of one NODE / PROJ op (bf16 storage only; every section starts 128-byte aligned):
 *   [0, Kp*C*2)          forward B operand: bf16 [Kp/8][C][8] = W[n][k] (k < Cin, zero padded to Kp = ceil16(Cin)),
 *                         eval mode: W[n][k] * gamma[n] / sqrt(running_var[n] + eps)
 *   then  float bias[C]   (eval: (b - running_mean) * gamma / sqrt(running_var + eps) + beta)
 *   then  float taps[9][C] (NODE only: depthwise weights, tap-major)
 *   then  (NODE, train)   backward B operand: bf16 [C/8][C][8] = W[o][i] stored as [o/8][i][o%8]
 * mmd_packed_bytes(kind, Cin, C) returns the block size the host must reserve. */
size_t mmd_packed_bytes(int32_t kind, int32_t Cin, int32_t C);

/* (Re)build the packed blocks of every NODE_FWD / PROJ_FWD op in `ops` whose `packed` reference is non-NULL, from the
 * current fp32 parameters (and, in eval mode, the running statistics).  One or two launches for a whole stack.  Call it
 * whenever the parameters may have changed since the last call (every training step; once for frozen teachers).
 * COPY ops of the list run first, for both dtypes.  An op with train = 0 that saves its depthwise output (save_d) is a
 * header that will be differentiated: its backward operand is packed as well.  The BatchNorm vector (out.bn) of every op
 * with frozen_bn = 1 is written here too, for both dtypes (bf16: by the packing launch, fp32: one launch of its own), so
 * a training forward with frozen layers must call this before mmd_bifpn_run / _run_multi with the same bases. */
int mmd_bifpn_prep(const MmdOp* ops, int32_t n_ops, void* const* bases, int32_t n_bases, int32_t C, int32_t dtype,
                   mmd_stream_t stream);

/* Run `n_ops` ops in order on `stream`.  `C` is the pyramid channel count (112 for EfficientDet-D2). */
int mmd_bifpn_run(const MmdOp* ops, int32_t n_ops, void* const* bases, int32_t n_bases,
                  int32_t B, int32_t C, int32_t dtype, mmd_stream_t stream);

/* Run `n_lists` op lists (e.g. the student's and the three teachers' forward) in lockstep on ONE stream: ops at the same
 * index that have the same kind and geometry share a launch (blockIdx.y = network), which matters for the small pyramid
 * levels (fewer tiles than SMs) and cuts the launch count by the number of networks; anything that does not line up
 * runs as in mmd_bifpn_run.  Every list must use the same batch size B.  n_lists <= 4. */
int mmd_bifpn_run_multi(const MmdOp* const* ops, const int32_t* n_ops, void* const* const* bases, const int32_t* n_bases,
                        int32_t n_lists, int32_t B, int32_t C, int32_t dtype, mmd_stream_t stream);

/* Optional profiler: while enabled, every kernel launch of this library is bracketed by a CUDA-event pair on its
 * stream.  mmd_prof_collect synchronises the device and ADDS, per kernel kind, the elapsed milliseconds, the number
 * of launches and the algorithmic bytes (DESIGN.md) into the caller's arrays of length mmd_prof_num_kinds(). */
void mmd_prof_enable(int on);
int mmd_prof_num_kinds(void);
const char* mmd_prof_kind_name(int kind);
int mmd_prof_collect(double* ms, long long* launches, double* algo_bytes);

/* Runtime switches of the library (process-wide; each also has an environment default that is read once):
 *   "chain_fwd"  0 / 1   run consecutive P5-P7 forward nodes of mmd_bifpn_run / _run_multi as ONE persistent launch with
 *                        grid barriers between the nodes (cooperative launch).  Default 0 (env MMD_CHAIN=1): measured
 *                        slower than separate launches on B200, see profiles/r2_chain_fwd.md.
 *   "mta_fast"   0 / 1   MTA pooling / backward of bf16 NHWC C = 112 p = 2 maps on the super-chunk kernels (7 fully coalesced
 *                        warp loads per 16 pixels) instead of the generic ones.  Default 1 (env MMD_NO_MTA_FAST=1 -> 0).
 *   "proj_tma"   0 / 1   first-cell projections (forward, bf16) on the warp-specialised tensor-map TMA pipeline
 *                        (cp.async.bulk.tensor loads / stores, double-buffered TMEM accumulator) instead of
 *                        proj_fwd_tc_kernel.  Default 1 (env MMD_NO_PROJ_TMA=1 -> 0).
 * Returns 0, or MMD_E_ARG for an unknown name. */
int mmd_set_option(const char* name, int32_t value);

/* sizeof(MmdOp) / sizeof(MmdMtaArgs) as compiled, so a binding can verify its struct mirror */
size_t mmd_sizeof_op(void);
size_t mmd_sizeof_mta_args(void);
size_t mmd_sizeof_focal_args(void);
size_t mmd_sizeof_pseudo_args(void);
size_t mmd_sizeof_adam_args(void);

#ifdef __cplusplus
}
#endif
#endif /* MMD_H */
