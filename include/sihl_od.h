/*
 * sihl_od.h — C ABI of libsihl_b200.so: the dense tail of sihl's ObjectDetection
 * head (anchor grid, CIoU top-k assignment, loss reductions + their backward,
 * top-k decode, dense decode + class-aware NMS) as hand-written sm_100a kernels.
 *
 * The reference (jonregef/sihl) is pure Python and has no FFI; its boundary for
 * this path is the `Head` protocol (ref: src/sihl/heads/__init__.py:28-53) as
 * implemented by `ObjectDetection` (ref: src/sihl/heads/object_detection.py).
 * Each entry point below names the reference lines it replaces.  The Python
 * host side (sihl_b200/heads/object_detection.py) binds these with ctypes; see
 * INTEGRATION.md for the stub a sihl maintainer would add.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer owned by the caller unless the name ends
 *    in `_host`; nothing is allocated, freed or retained by the library;
 *  - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *    every call only enqueues work on it and returns (no host synchronisation);
 *  - return value: 0 = SIHL_OD_OK, otherwise an error code; the message is
 *    available from sihl_od_last_error_string() (thread-local).  Nothing throws;
 *  - tensors are dense, row-major, fp32 unless stated; indices follow the
 *    reference: anchors are level-major, row-major (y outer, x inner), boxes
 *    are xyxy; ragged ground truth is CSR: gt_boxes [sumG,4], gt_classes
 *    [sumG] (int64), gt_offsets [B+1] (int32, device);
 *  - re-entrant: no global mutable state besides the thread-local error text.
 */
#ifndef SIHL_OD_H
#define SIHL_OD_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define SIHL_OD_API __attribute__((visibility("default")))
#else
#define SIHL_OD_API
#endif

#define SIHL_OD_OK      0
#define SIHL_OD_EINVAL  1   /* bad argument (mirrors the reference's asserts / torch errors) */
#define SIHL_OD_ECUDA   2   /* a CUDA runtime call failed */

#define SIHL_OD_MAX_LEVELS 8
#define SIHL_OD_MAX_TOPK   16
#define SIHL_OD_MAX_PEERS  16      /* GPUs of one node taking part in the fused loss-sum exchange */
#define SIHL_OD_IPC_HANDLE_BYTES 64
#define SIHL_OD_NUM_SUMS   8
#define SIHL_OD_MAX_BATCH_BY_VALUE 512  /* images whose gt counts sihl_od_train_assign can take from the host by value */

/* Element type of the head-output maps handed to the sihl_od_train_* and *_t entry points (the reference trains
 * with precision="16-mixed", ref examples/object_detection.py:294, and upcasts inside its autocast-off blocks,
 * ref object_detection.py:178,:195,:206): the kernels load this type and upcast in registers. */
#define SIHL_OD_F32  0
#define SIHL_OD_F16  1
#define SIHL_OD_BF16 2

/* Layout of the fp64 partial-sum vector every loss kernel accumulates into and
 * the one thing that crosses GPUs (one all-reduce of 8 doubles per step):
 *   [0] sum BCE-with-logits(loc, rel==1)      ref object_detection.py:160-162
 *   [1] #(rel == 1)                           ref :159,163
 *   [2] sum (iou_pred - rel)^2                ref :177-179
 *   [3] sum rel  (== sum of positive weights) ref :180,197,208
 *   [4] sum w * CIoU-loss(decoded box, gt)    ref :194-197
 *   [5] sum w * CE(class logits, gt class)    ref :205-208
 *   [6] #(rel > 0)  (P, number of positives)  ref :165,182
 *   [7] scratch: number of 32-row positive chunks published for
 *       sihl_od_pos_loss_tiles (not a loss term)                              */

SIHL_OD_API int sihl_od_version(void);
SIHL_OD_API const char *sihl_od_last_error_string(void);

/* ---- a1/a2: anchor grid ---------------------------------------------------
 * Replaces ObjectDetection.get_offsets_and_scales (ref :83-97) and the anchor
 * product (ref :134-140).  level_hw_host: HOST array [n_levels][2] = (h_l, w_l).
 * Outputs [A,4] each, A = sum h_l*w_l; any of them may be NULL. */
SIHL_OD_API int sihl_od_anchors(const int32_t *level_hw_host, int n_levels, int img_w, int img_h,
                    float *offsets, float *scales, float *anchors, void *stream);

/* ---- a3/a4: label assignment ----------------------------------------------
 * Replaces the per-image ObjectDetection.bbox_matching loop (ref :143-148,
 * :252-284; CIoU from torchvision ops/boxes.py:404-434) in two stages.
 *
 * Stage 1, select: per gt, the top-k anchors by clamp(CIoU,0) restricted to
 * positive values (ties: lowest anchor index), and the gt's best CIoU.
 *   level_hw_host != NULL: anchors must be the grid produced by sihl_od_anchors
 *     for these levels; candidates are enumerated from the gt extent (every
 *     anchor with CIoU > 0 overlaps the gt) and evaluated on the given table.
 *   level_hw_host == NULL: arbitrary anchors, all A x G pairs are evaluated.
 * anchor_terms (optional, may be NULL): [A,4] = (area, cx, cy, atan(w/h)) per anchor as
 * written by sihl_od_anchor_terms() — the per-anchor half of the CIoU hoisted out of the
 * pair loop (same fp32 operations, so results are unchanged) and cacheable with the tables.
 * Outputs: sel_anchor int32 [sumG, topk] (-1 = unused slot), sel_val fp32
 * [sumG, topk] (descending), best_iou fp32 [sumG].  If sums != NULL the 8
 * doubles are zeroed here (saves a memset launch per step).
 * Errors: topk outside 1..SIHL_OD_MAX_TOPK, A < topk with sumG > 0 (torch.topk
 * raises in the reference), n_levels > SIHL_OD_MAX_LEVELS, level sizes that do
 * not add up to A. */
SIHL_OD_API int sihl_od_anchor_terms(const float *anchors, int64_t num_anchors, float *terms, void *stream);

SIHL_OD_API int sihl_od_assign_select(const float *anchors, const float *anchor_terms, int64_t num_anchors,
                          const int32_t *level_hw_host, int n_levels, int img_w, int img_h,
                          const float *gt_boxes, const int32_t *gt_offsets, int batch, int total_gt,
                          int topk, int32_t *sel_anchor, float *sel_val, float *best_iou,
                          double *sums, void *stream);

/* Stage 2, resolve (+ fused dense losses): per anchor the maximum over the gts
 * that selected it (ties: lowest gt index, torch.max), relative IoU =
 * value / best_iou[gt] (relative != 0) or the value itself.
 *   assignment int64 [B,A]: gt index within the image, -1 where iou is not > 0
 *     (canonical form; the reference leaves implementation-defined indices on
 *     zero-IoU fill slots which nothing downstream reads, SURVEY.md §3.4);
 *   out_iou fp32 [B,A].
 * If loc_logits != NULL (and optionally iou_preds) the BCE / MSE reductions of
 * ref :157-163, :175-180 are accumulated into sums[0..3,6] in the same pass.
 * Positive lists (ref :182-184 order = row-major (b,a)): if tile_pos_count !=
 * NULL the kernel writes, per (image, tile), the number of positives and their
 * flat indices b*A+a in ascending order into tile_pos_rows [B * n_tiles * tile];
 * query the geometry with sihl_od_resolve_tiles().  sihl_od_pos_loss_tiles()
 * consumes the lists directly for dense maps (sihl_od_train_assign compacts them
 * into one pos_index for the reference's gathered-row MLPs).
 * prefetch_box_raw / prefetch_cls_logits (optional dense maps [B*A,4] / [B*A,C]):
 * the rows of the positives are prefetched into L2 for that next kernel.
 * pos_chunks (optional, int32 [B * n_tiles * tile / 32]): work list of 32-row chunks
 * of the positive lists for sihl_od_pos_loss_tiles; its length is kept in sums[7].
 * tile_pos_aux (optional, int32 [B * n_tiles * tile * 2]): per listed positive the
 * pair (global gt index, rel_iou bits), parallel to tile_pos_rows. */
SIHL_OD_API int sihl_od_resolve_tiles(int64_t num_anchors, int *n_tiles, int *tile);

SIHL_OD_API int sihl_od_assign_resolve(const int32_t *sel_anchor, const float *sel_val, const float *best_iou,
                           const int32_t *gt_offsets, int batch, int64_t num_anchors, int topk, int relative,
                           const float *loc_logits, const float *iou_preds,
                           int64_t *assignment, float *out_iou, double *sums,
                           int32_t *tile_pos_count, int32_t *tile_pos_rows,
                           const float *prefetch_box_raw, const float *prefetch_cls_logits, int num_classes,
                           int32_t *pos_chunks, int32_t *tile_pos_aux, void *stream);

/* The same entry for head-output maps of element type map_dtype (loc_logits, iou_preds and the two prefetch maps share
 * it): loaded as they are, upcast in registers.  For half types the BCE term follows the reference, which evaluates
 * log_sigmoid on the half logits (ref :160-161): it is rounded to the map type before entering the fp32 sum. */
SIHL_OD_API int sihl_od_assign_resolve_t(const int32_t *sel_anchor, const float *sel_val, const float *best_iou,
                           const int32_t *gt_offsets, int batch, int64_t num_anchors, int topk, int relative,
                           const void *loc_logits, const void *iou_preds, int map_dtype,
                           int64_t *assignment, float *out_iou, double *sums,
                           int32_t *tile_pos_count, int32_t *tile_pos_rows,
                           const void *prefetch_box_raw, const void *prefetch_cls_logits, int num_classes,
                           int32_t *pos_chunks, int32_t *tile_pos_aux, void *stream);

/* ---- N1 (SURVEY.md §8f): the un-clamped assignment of QuadrilateralDetection ---
 * ref: src/sihl/heads/quadrilateral_detection.py:266-294 (bbox_matching) and the
 * per-image loop :165-172, for a whole batch in two launches.  Arbitrary anchors
 * [A,4] (xyxy px), gt boxes in CSR form.  Every gt selects exactly topk anchors
 * by raw CIoU (no clamp; ties: lowest anchor); per anchor the maximum over the
 * selecting gts' values and one zero per non-selecting gt (ties: lowest gt).
 *   assignment int64 [B,A]: gt index within the image where rel_iou > 0, else -1
 *     (canonical: the reference stores the index of an arbitrary zero entry there
 *     and reads assignment only where rel_iou > 0, :188,:201);
 *   o2o_mask uint8 [B,A] (torch.bool storage): the anchor is some gt's best match;
 *   o2m_iou fp32 [B,A]; rel_iou fp32 [B,A] = nan_to_num(o2m_iou / best_iou[gt]).
 * Workspaces: sel_anchor int32 [sumG,topk], sel_val fp32 [sumG,topk] (the per-gt
 * top-k, descending — also an output), anchor_terms fp32 [A,4]. */
SIHL_OD_API int sihl_od_quad_matching(const float *anchors, int64_t num_anchors, const float *gt_boxes,
                          const int32_t *gt_offsets, int batch, int total_gt, int topk,
                          int64_t *assignment, uint8_t *o2o_mask, float *o2m_iou, float *rel_iou,
                          int32_t *sel_anchor, float *sel_val, float *anchor_terms, void *stream);

/* ---- a5-a10: losses ---------------------------------------------------------
 * Positive-row losses (ref :187-208; CIoU loss from torchvision
 * ops/ciou_loss.py:47-64, diou_loss.py:64-91, _utils.py:87-106) over DENSE maps
 * (box_raw [B*A,4], cls_logits [B*A,C]) taken straight from the per-tile lists of
 * sihl_od_assign_resolve: no compaction pass, no host round trip.  pos_chunks /
 * tile_pos_rows / tile_pos_aux are what sihl_od_assign_resolve published (the
 * chunk count lives in sums[7]).
 * Accumulates sums[4], sums[5].  If losses != NULL (with done_counter, a
 * zero-initialised uint32 the kernel resets itself) the last CTA also performs
 * sihl_od_loss_finalize — one launch less on a single GPU. */
SIHL_OD_API int sihl_od_pos_loss_tiles(const int32_t *pos_chunks, const int32_t *tile_pos_rows,
                           const int32_t *tile_pos_aux, int batch, int64_t num_anchors,
                           const float *offsets, const float *scales, int img_w, int img_h,
                           const float *gt_boxes, const int64_t *gt_classes, const int32_t *gt_offsets,
                           const float *box_raw, const float *cls_logits, int num_classes,
                           double *sums, float *losses, uint32_t *done_counter, void *stream);

/* ---- §8e: the one cross-GPU exchange, fused into the loss kernel ---------------
 * Same as sihl_od_pos_loss_tiles with losses / done_counter given, plus the
 * all-reduce (sum) of the 8 partial sums over the `world` GPUs of the node done
 * by the kernel's last CTA over peer memory (NVLink P2P stores + release/acquire
 * flags) before it finalizes: sums [8] then hold the global sums and losses the
 * global-batch losses (identical bits on every rank: contributions are added in
 * rank order) — no NCCL launch, no separate finalize launch.  peer_regions: DEVICE
 * array of `world` device pointers, entry r = rank r's exchange region as seen
 * from this process (own region at [rank]).  Every rank must launch the same
 * sequence of calls on a region — a shard without images (batch == 0) included:
 * it pushes zeros.  A peer that never arrives ends the wait after the region's
 * timeout (sihl_od_exchange_set_timeout; default 120 s) with NaN sums (no hang)
 * and the step number is latched in the region (sihl_od_exchange_status), so the
 * host can tell a timeout from a NaN loss.  world == 1 behaves like
 * sihl_od_pos_loss_tiles. */
SIHL_OD_API int sihl_od_pos_loss_tiles_exchange(const int32_t *pos_chunks, const int32_t *tile_pos_rows,
                           const int32_t *tile_pos_aux, int batch, int64_t num_anchors,
                           const float *offsets, const float *scales, int img_w, int img_h,
                           const float *gt_boxes, const int64_t *gt_classes, const int32_t *gt_offsets,
                           const float *box_raw, const float *cls_logits, int num_classes,
                           double *sums, float *losses, uint32_t *done_counter,
                           void *const *peer_regions, int world, int rank, void *stream);

/* ... and for dense maps of element type map_dtype (box_raw [B*A,4], cls_logits [B*A,C]).  Both maps may point into
 * PINNED HOST memory: the positives' rows are then gathered in place over PCIe (one warp instruction per class row when a
 * row has at most 32 16-byte vectors, the row read once, its raw box requested with it). */
SIHL_OD_API int sihl_od_pos_loss_tiles_exchange_t(const int32_t *pos_chunks, const int32_t *tile_pos_rows,
                           const int32_t *tile_pos_aux, int batch, int64_t num_anchors,
                           const float *offsets, const float *scales, int img_w, int img_h,
                           const float *gt_boxes, const int64_t *gt_classes, const int32_t *gt_offsets,
                           const void *box_raw, const void *cls_logits, int map_dtype, int num_classes,
                           double *sums, float *losses, uint32_t *done_counter,
                           void *const *peer_regions, int world, int rank, void *stream);

/* Exchange regions (one per step in flight), allocated in blocks and shared between
 * the per-GPU processes through CUDA IPC.  _create: cudaMalloc + zero a block of
 * n_regions regions of sihl_od_exchange_region_bytes(world) each and export its
 * handle (SIHL_OD_IPC_HANDLE_BYTES bytes, to be sent to the peers by any means,
 * e.g. torch.distributed.all_gather); _open maps a peer's block into this process
 * (peer access is enabled on first use); _close / _destroy undo them.  Not on the
 * per-step path. */
SIHL_OD_API size_t sihl_od_exchange_region_bytes(int world);
SIHL_OD_API int sihl_od_exchange_create(int world, int n_regions, void **block, unsigned char *ipc_handle_out);
SIHL_OD_API int sihl_od_exchange_open(const unsigned char *ipc_handle, void **peer_block);
SIHL_OD_API int sihl_od_exchange_close(void *peer_block);
SIHL_OD_API int sihl_od_exchange_destroy(void *block);
/* Per region (own block only; synchronous copies, not on the per-step path): the bound of the in-kernel wait in ns
 * (0 = default 120 s), and the sticky status: *timed_out_step = the first step whose wait ran out (0 = none),
 * *steps_done (may be NULL) = exchanges performed on this region so far. */
/* Device-side barrier over the node's GPUs on a region of its own (never one the fused exchange uses): enqueues one
 * tiny kernel that returns once every rank has enqueued — and the GPU reached — the same call.  Aligns the start of a
 * timed region across GPUs without a host barrier.  peer_regions as for sihl_od_pos_loss_tiles_exchange. */
SIHL_OD_API int sihl_od_exchange_barrier(void *const *peer_regions, int world, int rank, void *stream);
SIHL_OD_API int sihl_od_exchange_set_timeout(void *region, int world, uint64_t timeout_ns);
SIHL_OD_API int sihl_od_exchange_status(const void *region, int world, uint64_t *timed_out_step, uint64_t *steps_done);

/* ref :163-172, :180, :197, :208, :210 — losses fp32 [5] =
 * [location, box, class, iou, total]; early-out when sums[6] == 0. */
SIHL_OD_API int sihl_od_loss_finalize(const double *sums, float *losses, void *stream);

/* ---- the training step of the drop-in head, three calls (SURVEY.md §8f N2) ------------------
 * What ObjectDetection.training_step (ref :124-217) does around its MLPs, with no host
 * synchronisation, no allocation and a fixed launch sequence (CUDA-graph capturable):
 *
 *   sihl_od_train_assign   before the MLPs   ref :134-148 (+ :182-184 positive compaction)
 *   sihl_od_train_loss     after the MLPs    ref :157-217 (four losses + total, early-out on device)
 *   sihl_od_train_loss_bwd backward          SURVEY.md §7.4
 *
 * The number of positives P is only known on the device (pos_total).  The gathered-row MLPs of
 * the reference (box_head / cls_head on flat_feats[o2m_mask], ref :184-200) therefore run on a
 * STATIC number of rows pos_capacity >= P — min(topk * sumG, B * A) is always enough — of which
 * the kernels read / differentiate the first P only: pos_index[P..capacity) is filled with 0
 * (a valid row to gather) and the gradients of those rows are written as zeros.
 *
 * sihl_od_train_assign: select + resolve + compaction (3 launches).
 *   Ground truth: gt_boxes [gt_capacity,4] device; per-image counts EITHER as gt_counts_host
 *   (HOST int32 [batch], batch <= SIHL_OD_MAX_BATCH_BY_VALUE: passed to the kernel by value,
 *   which then also writes gt_offsets [batch+1] — no host->device copy, no sync) OR, with
 *   gt_counts_host == NULL, as gt_offsets [batch+1] already on the device (then the true total
 *   is read from gt_offsets[batch] on the device and gt_capacity only sizes the launch, so a
 *   captured graph can be replayed on new ground truth).
 *   Outputs: assignment int64 [B,A], rel_iou [B,A] (as sihl_od_assign_resolve, relative),
 *   pos_index int32 [pos_capacity] (flat b*A+a ascending = row order of flat_feats[o2m_mask],
 *   then zeros), pos_total int32 [1] (true P, may exceed pos_capacity: callers size it so that
 *   it cannot), sums [8] zeroed.  workspace: sihl_od_train_workspace_bytes(). */
SIHL_OD_API size_t sihl_od_train_workspace_bytes(int batch, int64_t num_anchors, int gt_capacity, int topk);

SIHL_OD_API int sihl_od_train_assign(const float *anchors, const float *anchor_terms, int64_t num_anchors,
                         const int32_t *level_hw_host, int n_levels, int img_w, int img_h,
                         const float *gt_boxes, const int32_t *gt_counts_host, int32_t *gt_offsets,
                         int batch, int gt_capacity, int topk,
                         int64_t *assignment, float *rel_iou,
                         int32_t *pos_index, int64_t pos_capacity, int32_t *pos_total,
                         double *sums, void *workspace, size_t workspace_bytes, void *stream);

/* sihl_od_train_loss: ONE launch for the four loss sums (dense BCE / MSE over [B*A], weighted
 * CIoU loss / cross-entropy over the first P compact rows) and — if losses != NULL — the five
 * losses [location, box, class, iou, total] written by the last CTA (ref :163-172 early-out
 * included).  losses == NULL leaves sums for an all-reduce + sihl_od_loss_finalize.
 * Maps of element type map_dtype: loc_logits [B*A], iou_preds [B*A], box_rows [pos_capacity,4],
 * cls_rows [pos_capacity,C].  For half types the location term reproduces the reference, which
 * evaluates log_sigmoid on the HALF logits (ref :160-161 has no .to(float32)): the per-element
 * log-sigmoid is rounded to the map type before it enters the fp32 sum.
 * A gt class outside [0, num_classes) makes the class loss NaN (torch raises a device assert).
 * sums must be the vector sihl_od_train_assign zeroed for this step (sums[7] is used as the
 * completion counter of the launch). */
SIHL_OD_API int sihl_od_train_loss(const void *loc_logits, const void *iou_preds, const void *box_rows, const void *cls_rows,
                       int map_dtype, int batch, int64_t num_anchors, int num_classes,
                       const float *rel_iou, const int64_t *assignment,
                       const int32_t *pos_index, int64_t pos_capacity, const int32_t *pos_total,
                       const float *offsets, const float *scales, int img_w, int img_h,
                       const float *gt_boxes, const int64_t *gt_classes, const int32_t *gt_offsets,
                       double *sums, float *losses, void *stream);

/* sihl_od_train_loss_bwd: ONE launch for all four gradients, written in map_dtype
 * (SURVEY.md §7.4).  grad_losses: device fp32 [5] = upstream gradient of [location, box,
 * class, iou, total] (NULL: d total = 1); the effective weights are
 * g_i = grad_losses[i] + grad_losses[4] * {1,10,1,1}[i] (ref :210), times grad_scale (1, or the
 * world size when the sums were all-reduced and DDP will average the gradients).  With
 * w = rel_iou of row r's location pos_index[r]:
 *   dloc[i]  = g0 * (sigmoid(loc) - [rel==1]) / sums[1]
 *   diou[i]  = g3 * 2 (iou_pred - rel) / sums[3]
 *   dcls_rows[r] = g2 * w/sums[3] * (softmax - onehot)   (NaN for a gt class outside [0, C))
 *   dbox_rows[r] = g1 * w/sums[3] * dCIoU/dpred * scales * exp(raw), the CIoU alpha held constant
 * dloc / diou [B*A]; dbox_rows [pos_capacity,4] / dcls_rows [pos_capacity,C]: rows >= P are
 * zeroed.  Any output may be NULL.  With no positives (sums[6] == 0) everything but dloc is zero
 * (the reference's early-out, ref :165-172, returns before the box / class / iou heads run). */
SIHL_OD_API int sihl_od_train_loss_bwd(const void *loc_logits, const void *iou_preds, const void *box_rows, const void *cls_rows,
                           int map_dtype, int batch, int64_t num_anchors, int num_classes,
                           const float *rel_iou, const int64_t *assignment,
                           const int32_t *pos_index, int64_t pos_capacity, const int32_t *pos_total,
                           const float *offsets, const float *scales, int img_w, int img_h,
                           const float *gt_boxes, const int64_t *gt_classes, const int32_t *gt_offsets,
                           const double *sums, const float *grad_losses, float grad_scale,
                           void *dloc, void *diou, void *dbox_rows, void *dcls_rows, void *stream);

/* ---- a11: forward tail ------------------------------------------------------
 * ref :108-109: per image the K largest location logits, sorted descending
 * (ties: lowest index).  idx int64 [B,K], top_logits fp32 [B,K]. */
SIHL_OD_API int sihl_od_topk(const float *loc_logits, int batch, int64_t num_anchors, int k,
                 int64_t *idx, float *top_logits, void *stream);

/* ref :113-121 on gathered rows: scores = sigmoid(top_logits), num_instances =
 * #(score > 0.5), classes = first argmax of cls_rows [B,K,C], boxes =
 * (offsets[idx] + scales[idx] * exp(box_rows)) * [W,H,W,H].
 * num_instances int64 [B], scores [B,K], classes int64 [B,K], boxes [B,K,4]. */
SIHL_OD_API int sihl_od_decode_rows(const float *top_logits, const int64_t *idx, int batch, int k,
                        const float *cls_rows, int num_classes, const float *box_rows,
                        const float *offsets, const float *scales, int img_w, int img_h,
                        int64_t *num_instances, float *scores, int64_t *classes, float *boxes,
                        void *stream);

/* The same two entry points for head outputs of element type map_dtype (SIHL_OD_F32 / _F16 / _BF16), loaded as
 * they are and upcast in registers.  top_logits stay fp32 (half values are exact in fp32).  For half maps
 * scores = sigmoid() and exp(raw box) are rounded to the map type before use, which is what the reference's
 * `.sigmoid()` / `.exp()` return under autocast (ref :113,:121), so num_instances and boxes follow it. */
SIHL_OD_API int sihl_od_topk_t(const void *loc_logits, int map_dtype, int batch, int64_t num_anchors, int k,
                   int64_t *idx, float *top_logits, void *stream);
SIHL_OD_API int sihl_od_decode_rows_t(const float *top_logits, const int64_t *idx, int batch, int k,
                          const void *cls_rows, int num_classes, const void *box_rows, int map_dtype,
                          const float *offsets, const float *scales, int img_w, int img_h,
                          int64_t *num_instances, float *scores, int64_t *classes, float *boxes,
                          void *stream);

/* ---- a15 (extension, not in the reference): dense decode + class-aware NMS --
 * Dense decode of every location: class = first argmax over C logits, score =
 * sigmoid(loc) (the semantics of ref :113,:117), candidate iff score >
 * score_thr, box decoded as ref :121.  Candidates are appended per image to
 * cand_* [B, cand_capacity] (unordered); cand_count int32 [B] must be zeroed by
 * the caller or by passing zero_counts != 0 (costs one tiny launch).
 * cand_key: uint64 [B,cap] sort key (score desc, location asc); cand_box
 * [B,cap,4]; cand_cls int32 [B,cap]. */
SIHL_OD_API int sihl_od_dense_decode(const float *loc_logits, const float *cls_logits, const float *box_raw,
                         int batch, int64_t num_anchors, int num_classes,
                         const float *offsets, const float *scales, int img_w, int img_h, float score_thr,
                         int32_t *cand_count, int64_t cand_capacity,
                         uint64_t *cand_key, float *cand_box, int32_t *cand_cls, int zero_counts,
                         void *stream);

/* sihl_od_dense_decode for maps of element type map_dtype (all three maps share it).  Half maps stream HALF the bytes
 * through the same TMA ring; scores and decoded boxes follow the reference's half semantics (sigmoid / exp rounded to
 * the map type, see sihl_od_decode_rows_t), so the candidate lists equal those of sihl_od_candidate_decode_t. */
SIHL_OD_API int sihl_od_dense_decode_t(const void *loc_logits, const void *cls_logits, const void *box_raw, int map_dtype,
                         int batch, int64_t num_anchors, int num_classes,
                         const float *offsets, const float *scales, int img_w, int img_h, float score_thr,
                         int32_t *cand_count, int64_t cand_capacity,
                         uint64_t *cand_key, float *cand_box, int32_t *cand_cls, int zero_counts,
                         void *stream);

/* Candidate-first variant of the same operation (same arguments, same outputs;
 * the candidate lists are unordered in both).  score = sigmoid(loc) does not
 * depend on the class logits (ref :113 vs :117), so the kernel streams only the
 * location map and gathers the class row + raw box of the locations that pass:
 * 4*A + n_cand*(4C+16) bytes read per image instead of 4*A*(C+5).  Preferred
 * while fewer than about half of the locations pass the threshold. */
SIHL_OD_API int sihl_od_candidate_decode(const float *loc_logits, const float *cls_logits, const float *box_raw,
                         int batch, int64_t num_anchors, int num_classes,
                         const float *offsets, const float *scales, int img_w, int img_h, float score_thr,
                         int32_t *cand_count, int64_t cand_capacity,
                         uint64_t *cand_key, float *cand_box, int32_t *cand_cls, int zero_counts,
                         void *stream);

/* sihl_od_candidate_decode for maps of element type map_dtype (all three maps share it).  cls_logits and box_raw may
 * point into PINNED HOST memory (cudaHostAlloc / cudaHostRegister, unified addressing): only the candidates' rows are then
 * read, in place, over PCIe — raw box and class row requested together; loc_logits must be device memory.  A PAGEABLE
 * host pointer is refused with SIHL_OD_EINVAL (it would fault in the kernel). */
SIHL_OD_API int sihl_od_candidate_decode_t(const void *loc_logits, const void *cls_logits, const void *box_raw, int map_dtype,
                         int batch, int64_t num_anchors, int num_classes,
                         const float *offsets, const float *scales, int img_w, int img_h, float score_thr,
                         int32_t *cand_count, int64_t cand_capacity,
                         uint64_t *cand_key, float *cand_box, int32_t *cand_cls, int zero_counts,
                         void *stream);

/* Class-aware greedy NMS per image over the candidate lists written by
 * sihl_od_dense_decode, semantics of torchvision _batched_nms_vanilla
 * (ops/boxes.py:102-120): visit by (score desc, location asc); a kept box
 * suppresses later boxes of the same class with IoU > iou_thr.  Emits the first
 * K kept detections per image, zero padded, in the reference forward()'s output
 * format.  workspace: sihl_od_nms_workspace_bytes(batch, cand_capacity) bytes (0 up to 256
 * candidates per image; NULL is then accepted): lists longer than 256 keep their working
 * arrays there, not in shared memory, so that the kernel fits on an SM beside the dense scan.
 * reset_counts != 0: cand_count[b] is zeroed once consumed, so the next
 * sihl_od_dense_decode needs no zeroing launch.
 * Precondition: the sort keys of a list are DISTINCT (every location listed at most once per image — what the decode
 * kernels write when cand_count started at zero).  Ranks are computed by counting; a list into which the same
 * candidates were appended twice (decode called again without zeroing the counters) is not a valid input. */
SIHL_OD_API size_t sihl_od_nms_workspace_bytes(int batch, int64_t cand_capacity);

SIHL_OD_API int sihl_od_nms_topk(const int32_t *cand_count, int64_t cand_capacity,
                     const uint64_t *cand_key, const float *cand_box, const int32_t *cand_cls,
                     int batch, float iou_thr, int k,
                     int64_t *num_instances, float *scores, int64_t *classes, float *boxes,
                     void *workspace, int reset_counts, void *stream);

/* The same operation for LONG candidate lists (thousands per image): suppression never
 * crosses classes, so every image's candidates are dealt to S = ceil(capacity / 2048)
 * (2..32) sub-lists by class, each sub-list is handled by its own CTA (S SMs per image,
 * sub-lists short enough for shared memory) and the image's K best are merged from the
 * S x K survivors.  Same results as sihl_od_nms_topk; three launches instead of one, so
 * the single-CTA entry stays the choice for the steady-state step with a few hundred
 * candidates per image.  workspace: sihl_od_nms_split_workspace_bytes(batch, capacity, k).
 * cand_count is consumed (zeroed when reset_counts != 0). */
SIHL_OD_API size_t sihl_od_nms_split_workspace_bytes(int batch, int64_t cand_capacity, int k);
SIHL_OD_API int sihl_od_nms_topk_split(int32_t *cand_count, int64_t cand_capacity, const uint64_t *cand_key,
                     const float *cand_box, const int32_t *cand_cls, int batch, float iou_thr, int k,
                     int64_t *num_instances, float *scores, int64_t *classes, float *boxes,
                     void *workspace, int reset_counts, void *stream);

/* Stand-alone batched NMS with torchvision.ops.batched_nms's signature, over
 * `n_images` independent segments: boxes [N,4], scores [N], classes int64 [N],
 * seg_offsets int32 [n_images+1] (device).  keep int64 [N]: per segment, the
 * kept indices (global, into [0,N)) in (score desc, index asc) order are
 * written at keep[seg_offsets[s] ...], keep_count int32 [n_images].
 * classes must lie in [0, 2^32).  workspace: sihl_od_batched_nms_workspace_bytes(N)
 * bytes (0 when every segment fits on chip; NULL is then accepted). */
SIHL_OD_API size_t sihl_od_batched_nms_workspace_bytes(int64_t n);

SIHL_OD_API int sihl_od_batched_nms(const float *boxes, const float *scores, const int64_t *classes,
                        const int32_t *seg_offsets, int n_images, int64_t n,
                        float iou_thr, int64_t *keep, int32_t *keep_count,
                        void *workspace, void *stream);

/* Class-aware DIoU-NMS (Zheng et al., "Distance-IoU Loss", AAAI 2020): the greedy NMS above with another suppression
 * test.  Visit by (score desc, location / index asc); a kept box i suppresses every later box j of the same class with
 *   diou(i, j) > diou_thr,  diou = iou - cd / diag  (torchvision's _box_diou_iou, eps = 1e-7), in fp32, in this order:
 *     w = max(0, min(x2_i, x2_j) - max(x1_i, x1_j)), h likewise;  inter = w * h
 *     iou = inter / ((area_i + area_j) - inter),  area = (x2 - x1) * (y2 - y1)
 *     wi = max(0, max(x2_i, x2_j) - min(x1_i, x1_j)), hi likewise;  diag = (wi * wi + hi * hi) + 1e-7
 *     dx = (x1_i + x2_i) / 2 - (x1_j + x2_j) / 2, dy likewise;  cd = dx * dx + dy * dy
 * so two strongly overlapping boxes with distinct centres (neighbouring objects in a crowd) can both survive.  diou lies
 * in (-1, 1]; any threshold is accepted, and a negative one also suppresses same-class boxes that do not overlap.  A NaN
 * diou (two zero-area boxes) never suppresses.  Each entry takes exactly the arguments of its greedy-NMS counterpart,
 * with the same preconditions, workspace query (sihl_od_nms_workspace_bytes, sihl_od_nms_split_workspace_bytes,
 * sihl_od_batched_nms_workspace_bytes), output layout and choice of kernels. */
SIHL_OD_API int sihl_od_diou_nms_topk(const int32_t *cand_count, int64_t cand_capacity,
                     const uint64_t *cand_key, const float *cand_box, const int32_t *cand_cls,
                     int batch, float diou_thr, int k,
                     int64_t *num_instances, float *scores, int64_t *classes, float *boxes,
                     void *workspace, int reset_counts, void *stream);
SIHL_OD_API int sihl_od_diou_nms_topk_split(int32_t *cand_count, int64_t cand_capacity, const uint64_t *cand_key,
                     const float *cand_box, const int32_t *cand_cls, int batch, float diou_thr, int k,
                     int64_t *num_instances, float *scores, int64_t *classes, float *boxes,
                     void *workspace, int reset_counts, void *stream);
SIHL_OD_API int sihl_od_batched_diou_nms(const float *boxes, const float *scores, const int64_t *classes,
                        const int32_t *seg_offsets, int n_images, int64_t n,
                        float diou_thr, int64_t *keep, int32_t *keep_count,
                        void *workspace, void *stream);

/* Class-aware greedy NMS over quadrilaterals (text lines, documents, oriented objects; mmcv's nms_quadri) with the
 * contract of sihl_od_batched_nms: quads [N, 4, 2] fp32 (four points (x, y) in pixels, finite), scores [N], classes
 * int64 [N] in [0, 2^32), seg_offsets int32 [n_images+1] (device).  Per segment, visit by (score desc, index asc); a
 * kept quad i suppresses every later quad j of its class with quad_iou(i, j) > iou_thr.  keep / keep_count as in
 * sihl_od_batched_nms.  quad_iou is the IoU of the CONVEX HULLS of the two vertex sets, in fp32:
 *   - for convex quads the polygon IoU, whatever the start vertex and orientation (CW or CCW); bit-identical under any
 *     permutation of a quad's vertices; non-convex or self-intersecting vertex orders are taken by their hull;
 *   - 0 when either hull has zero area (collinear or repeated points) and when the AABBs do not overlap (an overlap of
 *     zero width counts as none);
 *   - inter clamped to [0, min(area_i, area_j)], iou = inter / ((area_i + area_j) - inter), 0 unless the union > 0;
 *   - quad_iou(i, j) and quad_iou(j, i) are the same bits.
 * So a negative iou_thr also suppresses same-class quads that do not overlap.  At most 90 000 quads per call (the
 * suppression mask takes up to N^2/64 words): larger n returns SIHL_OD_EINVAL.  Every n runs the whole-GPU bitmask
 * path; many segments go in one call.  workspace: sihl_od_batched_quad_nms_workspace_bytes(n) bytes (0 for n = 0, when
 * NULL is accepted; 0 as well for n outside [0, 90 000]).  No host synchronisation: the call can be captured in a
 * CUDA graph. */
SIHL_OD_API size_t sihl_od_batched_quad_nms_workspace_bytes(int64_t n);
SIHL_OD_API int sihl_od_batched_quad_nms(const float *quads, const float *scores, const int64_t *classes,
                        const int32_t *seg_offsets, int n_images, int64_t n,
                        float iou_thr, int64_t *keep, int32_t *keep_count,
                        void *workspace, void *stream);

/* out[i * nb + j] = quad_iou(a_i, b_j) (the overlap above) for quads a [na, 4, 2] and b [nb, 4, 2], fp32 [na, nb]
 * (device), one thread per pair; na * nb <= 2^38. */
SIHL_OD_API int sihl_od_quad_iou(const float *a, int64_t na, const float *b, int64_t nb, float *out, void *stream);

/* Class-aware box voting (merge-NMS; Gidaris & Komodakis, ICCV 2015; YOLOv5's non_max_suppression(merge=True)), one
 * pass after a greedy NMS (IoU or DIoU) that moves the coordinates of the kept boxes only.  For every emitted
 * detection k of class c, with the overlap and the threshold of the selection it follows (iou_thr / diou_thr):
 *   V_k  = { j in the same list : cls_j == c  and  overlap(b_k, b_j) > thr }   any rank, kept or suppressed, k included
 *   b'_k = sum_{j in V_k} s_j * b_j / sum_{j in V_k} s_j                       per coordinate
 * overlap is the IoU of sihl_od_nms_topk (the *_box_vote_* entries) or the diou of sihl_od_diou_nms_topk (the
 * *_diou_box_vote_* entries), in the same fp32 operator order; a NaN overlap never joins a cluster, and a negative
 * DIoU threshold admits same-class boxes that do not overlap.  s_j is the candidate's score (the high word of cand_key,
 * or scores[j]).  Every product s_j * x_j is exact in fp64; the sums are fp64 (their order is unspecified) and the
 * quotient is rounded once to fp32.  When V_k is empty or its score sum is 0 (thr >= 1, a zero-area kept box, scores
 * that underflow), b_k is left as it is.  Counts, scores, classes, keep indices and their order are not touched.
 * No workspace, no host synchronisation: the pass can be captured in a CUDA graph.
 *
 * Top-K entries: the candidate lists and the outputs of sihl_od_nms_topk / _split (or the DIoU entries) called with
 * reset_counts = 0, which leaves the lists and cand_count as they were; boxes [batch, k, 4] is rewritten in place,
 * rows past num_instances[b] (the zero padding) are not touched.  Batched entries: the inputs of sihl_od_batched_nms
 * (or sihl_od_batched_diou_nms) and its keep / keep_count; voted_boxes [N, 4] receives the voted box of keep[i] at row
 * i for the first keep_count[s] positions of every segment and nothing elsewhere. */
SIHL_OD_API int sihl_od_box_vote_topk(const int32_t *cand_count, int64_t cand_capacity, const uint64_t *cand_key,
                     const float *cand_box, const int32_t *cand_cls, int batch, float iou_thr, int k,
                     const int64_t *num_instances, const int64_t *classes, float *boxes, void *stream);
SIHL_OD_API int sihl_od_diou_box_vote_topk(const int32_t *cand_count, int64_t cand_capacity, const uint64_t *cand_key,
                     const float *cand_box, const int32_t *cand_cls, int batch, float diou_thr, int k,
                     const int64_t *num_instances, const int64_t *classes, float *boxes, void *stream);
SIHL_OD_API int sihl_od_batched_box_vote(const float *boxes, const float *scores, const int64_t *classes,
                        const int32_t *seg_offsets, int n_images, int64_t n, float iou_thr,
                        const int64_t *keep, const int32_t *keep_count, float *voted_boxes, void *stream);
SIHL_OD_API int sihl_od_batched_diou_box_vote(const float *boxes, const float *scores, const int64_t *classes,
                        const int32_t *seg_offsets, int n_images, int64_t n, float diou_thr,
                        const int64_t *keep, const int32_t *keep_count, float *voted_boxes, void *stream);

/* Class-aware Soft-NMS (Bodla et al., ICCV 2017, Algorithm 1; mmcv's soft_nms) per image.  Scores are decayed
 * instead of dropped: starting from the candidates with score >= score_thr, repeatedly select the alive candidate
 * with the largest current score (ties: lowest location, or lowest input index for the stand-alone entry), emit it
 * with its current score, and multiply the score of every alive candidate of the SAME class by w(iou) where
 * iou = inter / ((area_m + area_j) - inter) in fp32 (the operator order of the hard NMS; NaN -> 0):
 *   SIHL_OD_SOFT_NMS_LINEAR:   w = iou > iou_thr ? 1 - iou : 1                           (fp32)
 *   SIHL_OD_SOFT_NMS_GAUSSIAN: w = (float)exp(-(double)iou * (double)iou / (double)sigma) (fp64 exp, one rounding)
 * A candidate whose decayed score falls below score_thr (or is NaN) is dropped.  Emitted scores never increase
 * along the output and are never below score_thr.  iou_thr is only read by the linear method, sigma (> 0) only by
 * the Gaussian one. */
#define SIHL_OD_SOFT_NMS_LINEAR 1
#define SIHL_OD_SOFT_NMS_GAUSSIAN 2

/* Soft-NMS over the candidate lists of sihl_od_dense_decode: same preconditions (distinct keys), output layout
 * (first K detections per image, zero padded past num_instances) and reset_counts meaning as sihl_od_nms_topk.
 * workspace: sihl_od_soft_nms_workspace_bytes(batch, cand_capacity) bytes (0 up to 32768 candidates per image, which
 * stay in shared memory; NULL is then accepted). */
SIHL_OD_API size_t sihl_od_soft_nms_workspace_bytes(int batch, int64_t cand_capacity);
SIHL_OD_API int sihl_od_soft_nms_topk(const int32_t *cand_count, int64_t cand_capacity,
                     const uint64_t *cand_key, const float *cand_box, const int32_t *cand_cls,
                     int batch, int method, float iou_thr, float sigma, float score_thr, int k,
                     int64_t *num_instances, float *scores, int64_t *classes, float *boxes,
                     void *workspace, int reset_counts, void *stream);

/* Segment form of the same operation, beside sihl_od_batched_nms: boxes [N,4], scores [N], classes int64 [N] in
 * [0, 2^32), seg_offsets int32 [n_images+1] (device).  Per segment s, at most max_out kept input indices (global, into
 * [0,N)) in selection order and their decayed scores are written at keep[seg_offsets[s] ...] and
 * keep_scores[seg_offsets[s] ...]; keep_count int32 [n_images].  Entries past keep_count are left untouched.
 * workspace: sihl_od_batched_soft_nms_workspace_bytes(N) bytes (0 up to N = 32768; NULL is then accepted). */
SIHL_OD_API size_t sihl_od_batched_soft_nms_workspace_bytes(int64_t n);
SIHL_OD_API int sihl_od_batched_soft_nms(const float *boxes, const float *scores, const int64_t *classes,
                        const int32_t *seg_offsets, int n_images, int64_t n,
                        int method, float iou_thr, float sigma, float score_thr, int max_out,
                        int64_t *keep, float *keep_scores, int32_t *keep_count,
                        void *workspace, void *stream);

/* ---- N3 (SURVEY.md §8f): detection <-> ground-truth matching for the validation mAP ----------
 * What torchmetrics' MeanAveragePrecision (ref object_detection.py:219-237, :245; COCOeval.evaluateImg of its
 * faster_coco_eval backend) does per image on the CPU at epoch end, done on the GPU right after forward():
 * detections [B,K] (boxes xyxy px, scores, classes int64 — all K rows of forward()'s output, as the reference passes
 * them) are ranked by (score desc, input order) and greedily matched per category to the CSR ground truth at
 * n_thresholds IoU thresholds and n_areas area ranges [lo, hi] (px^2; a gt outside the range is "ignored" and only
 * matched while no regular gt fits; an unmatched detection outside the range is ignored).  Box IoU in fp64.
 * HOST arrays: iou_thresholds_host [n_thresholds], area_ranges_host [n_areas][2].
 * Outputs: det_order int32 [B,K] (rank -> detection), dt_match int32 [B,n_areas,n_thresholds,K] by rank (global gt
 * index or -1), dt_ignore uint8 (same shape), gt_ignore uint8 [n_areas, total_gt].
 * workspace: sihl_od_map_workspace_bytes().  torchmetrics / faster_coco_eval are absent here: parity UNPINNED. */
SIHL_OD_API size_t sihl_od_map_workspace_bytes(int total_gt, int n_thresholds, int n_areas);
SIHL_OD_API int sihl_od_map_match(const float *det_boxes, const float *det_scores, const int64_t *det_classes, int batch, int k,
                      const float *gt_boxes, const int64_t *gt_classes, const int32_t *gt_offsets, int total_gt,
                      const double *iou_thresholds_host, int n_thresholds, const double *area_ranges_host, int n_areas,
                      int32_t *det_order, int32_t *dt_match, uint8_t *dt_ignore, uint8_t *gt_ignore,
                      void *workspace, void *stream);

/* The same matching for quadrilateral detections (the QuadrilateralDetection head): det_quads [B,K,8] and gt_quads
 * [total_gt,8] are four points (x, y) in px each, everything else and every output as sihl_od_map_match, in the same
 * layouts and under the same COCOeval.evaluateImg rule.  Two values change:
 *   iou(d, g)  = the IoU of the convex hulls of the two vertex sets, the fp32 value of sihl_od_quad_iou (bit-identical
 *                under any vertex order, 0 for disjoint AABBs or a zero-area hull), widened to double;
 *   area(q)    = the hull's polygon area in fp32, widened to double, for gts and unmatched detections alike (not the
 *                AABB's w * h: a thin slanted quad falls in the area range of its polygon).
 * The hulls are built once per quad and the same-class IoUs of each image are filled into a [K, G_b] matrix over the
 * whole GPU before the chains run.  K <= 1024, n_thresholds <= 16, n_areas <= 8.  workspace: at least
 * sihl_od_quad_map_workspace_bytes(batch, k, total_gt, n_thresholds, n_areas) bytes (that query returns 0 for
 * arguments out of range), passed in workspace_bytes; a shorter one is SIHL_OD_EINVAL.  batch = 0 reads and writes
 * nothing (its empty arrays may be NULL).  No host synchronisation: the call can be captured in a CUDA graph. */
SIHL_OD_API size_t sihl_od_quad_map_workspace_bytes(int batch, int k, int total_gt, int n_thresholds, int n_areas);
SIHL_OD_API int sihl_od_quad_map_match(const float *det_quads, const float *det_scores, const int64_t *det_classes,
                      int batch, int k, const float *gt_quads, const int64_t *gt_classes, const int32_t *gt_offsets,
                      int total_gt, const double *iou_thresholds_host, int n_thresholds, const double *area_ranges_host,
                      int n_areas, int32_t *det_order, int32_t *dt_match, uint8_t *dt_ignore, uint8_t *gt_ignore,
                      void *workspace, size_t workspace_bytes, void *stream);

/* The two matchings above with COCO's optional ground-truth annotations (COCOeval's iscrowd and area; computeIoU's
 * maskUtils.iou(d, g, iscrowd) and evaluateImg).  Arguments, limits, workspace query, argument checks and outputs are
 * those of the sibling entry, plus two DEVICE arrays [total_gt], either of which may be NULL (none: all zero):
 *   gt_crowd uint8  nonzero marks a crowd region ("don't care" in text datasets)
 *   gt_area  double the annotated area of the gt
 * Rules:
 *   1. a gt's area for the range test is gt_area[g] when gt_area[g] > 0; otherwise (<= 0, NaN, NULL) the sibling's
 *      (box: fp32 w and h multiplied in double; quad: the hull area widened).  Detections always use their own area.
 *   2. a crowd gt is ignored in every area range: gt_ignore[a, g] = crowd[g] || area outside range a.
 *   3. the overlap of a detection with a crowd gt is the intersection over the DETECTION's area (IoA): for boxes
 *      bbIou with u = the detection's w * h in fp64, with the IoU's early-outs; for quads the clamped hull intersection
 *      over the detection's hull area in fp32, widened, 0 for disjoint AABBs or a zero-area hull.  Non-crowd pairs get
 *      the sibling's IoU, bit for bit.
 *   4. a crowd gt is never taken: later detections may match it again at the same threshold.  Everything else in the
 *      chain is the sibling's (regular gts first, ignored ones only while nothing matched; the later of equal overlaps
 *      wins; the start min(t, 1 - 1e-10)).
 *   5. a detection matched to a crowd gt has dt_match = that gt's global index and dt_ignore = 1.
 * So crowd gts leave the recall denominator through gt_ignore and their detections the precision through dt_ignore.
 * With both pointers NULL the call computes exactly its sibling's tables.  batch = 0 reads and writes nothing (its empty
 * arrays may be NULL), for boxes as well.  No host synchronisation: the call can be captured in a CUDA graph.  torchmetrics / pycocotools are absent here: parity UNPINNED. */
SIHL_OD_API int sihl_od_map_match_crowd(const float *det_boxes, const float *det_scores, const int64_t *det_classes,
                      int batch, int k, const float *gt_boxes, const int64_t *gt_classes, const int32_t *gt_offsets,
                      int total_gt, const uint8_t *gt_crowd, const double *gt_area, const double *iou_thresholds_host,
                      int n_thresholds, const double *area_ranges_host, int n_areas, int32_t *det_order,
                      int32_t *dt_match, uint8_t *dt_ignore, uint8_t *gt_ignore, void *workspace, void *stream);
SIHL_OD_API int sihl_od_quad_map_match_crowd(const float *det_quads, const float *det_scores, const int64_t *det_classes,
                      int batch, int k, const float *gt_quads, const int64_t *gt_classes, const int32_t *gt_offsets,
                      int total_gt, const uint8_t *gt_crowd, const double *gt_area, const double *iou_thresholds_host,
                      int n_thresholds, const double *area_ranges_host, int n_areas, int32_t *det_order,
                      int32_t *dt_match, uint8_t *dt_ignore, uint8_t *gt_ignore, void *workspace,
                      size_t workspace_bytes, void *stream);

/* ---- N4 (SURVEY.md §8f): the per-location MLP towers in front of the hot path ----------------
 * ref object_detection.py:51-61 builds loc / cls / box / iou heads as torchvision ops.MLP(256 -> [256]*num_layers
 * + [out], norm_layer=LayerNorm, activation_layer=SiLU) and applies them to every location (:116, :121, :175).
 * One call = one layer over M locations, bf16 operands on the 5th-generation tensor cores (tcgen05.mma, fp32
 * accumulators in TMEM, operands staged by TMA), the whole Linear -> LayerNorm -> SiLU chain in one kernel:
 *   sihl_od_mlp_hidden: y = SiLU(LayerNorm(x W^T + bias; eps) * gamma + beta)   x [M,256], W [256,256], y [M,256] bf16
 *   sihl_od_mlp_out:    y = x W^T + bias       W [n_pad,256] bf16 (rows >= out_cols zero), y [M,out_cols] fp32
 * channels must be 256 (the reference's num_channels default); n_pad in {16,32,64,96,128,256}; bias/gamma/beta are
 * fp32 device arrays of length 256 (hidden) or n_pad (out).  x, W, y: device pointers, 16-byte aligned, row-major,
 * contiguous.  Inference only (no gradient is produced): training keeps torch's MLP. */
SIHL_OD_API int sihl_od_mlp_hidden(const void *x_bf16, int64_t m, int channels, const void *w_bf16, const float *bias,
                       const float *gamma, const float *beta, float eps, void *y_bf16, void *stream);
SIHL_OD_API int sihl_od_mlp_out(const void *x_bf16, int64_t m, int channels, const void *w_bf16, const float *bias,
                    int n_pad, int out_cols, float *y, void *stream);

/* Training path of a hidden layer (bf16 mixed precision, like autocast): the forward additionally stores every row's
 * LayerNorm statistics, row_stats [M,2] = (mean, rstd), and — when v_bf16 is given — the pre-activation v = x W^T + bias
 * (bf16 [M,256]; otherwise the caller recomputes it with sihl_od_lateral_linear(rows = x, identity row map)).  The backward
 * of LayerNorm + SiLU is one kernel over rows (v, dy streamed through a shared-memory ring by cp.async.bulk): v, dy ->
 * dv [M,256] bf16 and per-CTA partial column sums partials [partial_rows,3,256] fp32 = (d gamma, d beta, d bias), to be
 * summed over partial_rows (sihl_od_mlp_hidden_bwd_partial_rows() is the grid the kernel is tuned for).  The two gradient
 * GEMMs are plain matrix products: dx = dv W (sihl_od_lateral_linear with W^T, zero bias) and dW = dv^T x (library GEMM). */
SIHL_OD_API int sihl_od_mlp_hidden_train(const void *x_bf16, int64_t m, int channels, const void *w_bf16, const float *bias,
                             const float *gamma, const float *beta, float eps, void *y_bf16, float *row_stats,
                             void *v_bf16 /* optional: bf16 [M,256], the pre-activation, stored by the same epilogue so
                                             that the backward does not have to recompute it */,
                             void *stream);
SIHL_OD_API int sihl_od_mlp_bwd_partial_rows(void);
/* Grid (= rows of partials) the two sihl_od_mlp_hidden_bwd* entries are tuned for: two persistent CTAs per SM, each
 * streaming its rows through a shared-memory ring (cp.async.bulk + mbarrier).  They accept any partial_rows in
 * [1, sihl_od_mlp_bwd_partial_rows()] and write exactly that many rows of partials. */
SIHL_OD_API int sihl_od_mlp_hidden_bwd_partial_rows(void);
/* bf16 -> fp32 of n contiguous values (n % 8 == 0): the towers' input gradient handed back to the fp32 laterals. */
SIHL_OD_API int sihl_od_bf16_to_f32(const void *src_bf16, int64_t n, float *dst, void *stream);
SIHL_OD_API int sihl_od_mlp_hidden_bwd(const void *v_bf16, const void *dy_bf16, const float *row_stats, const float *gamma,
                           const float *beta, int64_t m, int channels, void *dv_bf16, float *partials,
                           int partial_rows, void *stream);
/* The same backward for a tower's LAST hidden layer when the Linear behind it has one output (the location and IoU towers,
 * ref object_detection.py:56, :60): the upstream gradient is the outer product dy[m,:] = bf16(dout[m]) * w_out[:] (dout fp32
 * [m] = gradient of the tower's output, w_out bf16 [256] = that Linear's weight row), formed in registers instead of being
 * materialised as an [M,256] matrix by a K = 1 library GEMM and read back. */
SIHL_OD_API int sihl_od_mlp_hidden_bwd_rank1(const void *v_bf16, const float *dout, const void *w_out_bf16, const float *row_stats,
                                 const float *gamma, const float *beta, int64_t m, int channels, void *dv_bf16,
                                 float *partials, int partial_rows, void *stream);

/* The laterals in front of the towers (ref object_detection.py:52-55, :102-105): Conv2dNormActivation(C_in, 256, 1,
 * activation_layer=None) = 1x1 conv + BatchNorm, per level, then "b c h w -> b (h w) c" and the concatenation over
 * the levels.  Inference (BatchNorm folded into weight and bias by the caller), C_in == 256:
 *   sihl_od_lateral_rows:   x [B, C, HW] fp32 (NCHW level) -> rows [B*HW, C] bf16   (C % 64 == 0)
 *   sihl_od_lateral_linear: y = rows W^T + bias on the tensor cores (same kernel family as the towers), bf16, row
 *       m = b*rows_per_image + i written at row b*out_rows_per_image + out_row_offset + i of y [B*out_rows_per_image, 256]:
 *       every level lands directly in its slice of the concatenated [B, A, 256] feature tensor the towers read. */
SIHL_OD_API int sihl_od_lateral_rows(const float *x_nchw, int batch, int channels, int64_t hw, void *rows_bf16, void *stream);
/* Training path of a lateral (batch-statistics BatchNorm, bf16 mixed precision).  Forward: the batch statistics of the
 * conv output follow from the input's first and second moments (mean = W s / M, E[y^2] = diag(W G W^T) / M with s = sum of
 * rows, G = rows^T rows), so the conv + BatchNorm is again ONE folded sihl_od_lateral_linear pass.  Backward over rows
 * [M,256] bf16 with n = the normalised conv output (recomputed with sihl_od_lateral_linear):
 *   sihl_od_bn_bwd_colsums: partials [partial_rows,2,256] = per-CTA sums over rows of (dz, dz*n)
 *   sihl_od_bn_bwd_apply:   dy = scale * (dz - mean_dz - n * mean_dzn)
 *   sihl_od_rows_to_nchw:   rows [B*HW, C] bf16 -> x [B, C, HW] fp32 (the input gradient handed back to the neck) */
SIHL_OD_API int sihl_od_bn_bwd_colsums(const void *dz_bf16, const void *n_bf16, int64_t m, int channels, float *partials,
                           int partial_rows, void *stream);
SIHL_OD_API int sihl_od_bn_bwd_apply(const void *dz_bf16, const void *n_bf16, const float *scale, const float *mean_dz,
                         const float *mean_dzn, int64_t m, int channels, void *dy_bf16, void *stream);
/* _map variants: dz is one level's slice of the gradient of the concatenated [B, dz_rows_per_image, 256] features, read in
 * place — row m of the level is row (m / rows_per_image) * dz_rows_per_image + dz_row_offset + m % rows_per_image of dz. */
SIHL_OD_API int sihl_od_bn_bwd_colsums_map(const void *dz_bf16, int64_t rows_per_image, int64_t dz_rows_per_image,
                               int64_t dz_row_offset, const void *n_bf16, int64_t m, int channels, float *partials,
                               int partial_rows, void *stream);
SIHL_OD_API int sihl_od_bn_bwd_apply_map(const void *dz_bf16, int64_t rows_per_image, int64_t dz_rows_per_image,
                             int64_t dz_row_offset, const void *n_bf16, const float *scale, const float *mean_dz,
                             const float *mean_dzn, int64_t m, int channels, void *dy_bf16, void *stream);
/* Column sums of bf16 rows [m,256] in fp32 — the first moment s of a lateral's input (see above): per-CTA partials
 * [partial_rows,256], partial_rows = sihl_od_mlp_bwd_partial_rows(), summed by the caller. */
SIHL_OD_API int sihl_od_rows_colsum(const void *rows_bf16, int64_t m, int channels, float *partials, int partial_rows,
                        void *stream);
SIHL_OD_API int sihl_od_rows_to_nchw(const void *rows_bf16, int batch, int channels, int64_t hw, float *x_nchw, void *stream);
SIHL_OD_API int sihl_od_lateral_linear(const void *rows_bf16, int64_t m, int channels, const void *w_bf16, const float *bias,
                           int64_t rows_per_image, int64_t out_rows_per_image, int64_t out_row_offset,
                           void *y_bf16, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* SIHL_OD_H */
