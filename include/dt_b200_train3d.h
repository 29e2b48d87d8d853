/* dt_b200_train3d.h — the training-step entry points of the single-level 3-D tube model (the R18-3D keypoint R-CNN of
 * configs/video/3d/03_R-18-3D_PTFromCOCO.yaml) in libdt_b200.so.  Same conventions as include/dt_b200.h: device pointers,
 * sizes and a stream; nothing allocated or synchronised inside; every argument validated on the host before any CUDA call;
 * 0 on success, otherwise dt_last_error() holds the message.  Bound in python by _lib.TRAIN3D_SIGNATURES. */
#ifndef DT_B200_TRAIN3D_H_
#define DT_B200_TRAIN3D_H_
#include "dt_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Tube RPN losses and their gradient (lib/modeling/model_builder.py:500-563 add_rpn_outputs(nd=True) and :612-635
 * add_rpn_losses(time_dim=T)) from the PER-FRAME head output out [B, T, H, W, ld_o] fp32 = [A logits | 4A deltas (a*4+k)]
 * per frame.  cls: the logits averaged over T (TimePool avg), Detectron SigmoidCrossEntropyLoss with its default
 * normalize=1: sum over labels >= 0, divided by max(#labels >= 0, 1e-5) over the whole labels [B, H, W, A] blob (counted
 * on the device into normalizer [1] fp32, a caller-provided scratch word), times scale_cls = 1 / NUM_GPUS.  bbox:
 * SmoothL1Loss(beta) against targets / inside_w / outside_w [B, H, W, 4TA] whose column a*4T + t*4 + k is channel a*4+k
 * of frame t (the layout of dt_rpn_targets), scale_box = 1 / NUM_GPUS / T / B.  grad [B, T, H, W, ld_g] bf16 in the
 * per-frame layout, padding 0; each frame carries logit gradient / T (the TimePool backward).  loss (may be NULL) [2]
 * fp32 += (cls, bbox). */
int dt_rpn_tube_loss_grad(const float* out, int ld_o, const int* labels, const float* targets, const float* inside_w,
                          const float* outside_w, int B, int T, int H, int W, int A, float scale_cls, float scale_box, float beta,
                          float* normalizer, void* grad, int ld_g, float* loss, void* stream);

/* dt_frcnn_loss_grad for the tube box head (model_builder.py:426-493 with time_dim = T): out [R*T, ld_o] fp32 holds the
 * per-RoI-frame rows of the fused cls_score_1 | bbox_pred_1 product, RoI r in rows r*T .. r*T+T-1.  The fold of
 * dt_fold_tube_heads (class logits = mean over the frames, box column c*4T + t*4 + k = channel C + c*4 + k of frame t) is
 * applied before the losses, its backward fused into the gradient: grad [R*T, ld_g] bf16 per RoI-frame, padding 0.
 * labels [R]; targets / inside_w / outside_w [R, 4CT]; scale_box = 1 / NUM_GPUS / T.  Loss, accuracy and the live-row
 * normalisation totals[0] as dt_frcnn_loss_grad, which is this function at T = 1. */
int dt_frcnn_tube_loss_grad(const float* out, int ld_o, const int* labels, const float* targets, const float* inside_w,
                            const float* outside_w, int R, int T, int C, const float* totals, float scale_cls, float scale_box,
                            void* grad, int ld_g, float* loss, float* accuracy, void* stream);

/* Backward of the res5 RoI head's two ReduceBackMeans (W, then H): out [N, H, W, C] bf16 = g [N, C] bf16 / (H*W), fused
 * with the pointwise step after it exactly like dt_bwd_pointwise2: masked by [y > 0] (y [N, H, W, C], may be NULL) and
 * scaled by scale[C] (may be NULL); out2 (may be NULL) receives the same masked value times scale2 (or unscaled). */
int dt_spatial_mean_bwd(const void* g, long long N, int H, int W, int C, const void* y, const float* scale, void* out,
                        const float* scale2, void* out2, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DT_B200_TRAIN3D_H_ */
