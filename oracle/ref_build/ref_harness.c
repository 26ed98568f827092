/*
 * TEST INFRASTRUCTURE -- not part of the product.  Only tests/, bench.py's
 * cpu_baseline / --impl reference legs and __graft_entry__.smoke() may load
 * the library this file builds (oracle/_ref/libtf_ref.so).
 *
 * Harness around the UNMODIFIED reference temporal filter.  It #includes
 * av1/encoder/temporal_filter.c where it lies under /root/reference (no source
 * is copied into this repo) so that the file-static functions
 * (tf_motion_search :87, tf_build_predictor :328, tf_normalize_filtered_frame
 * :740) become callable, fills the handful of AV1_COMP fields that
 * av1_tf_do_filtering_row (:788) reads, and runs the reference row by row.
 *
 * A hook is slipped in through the rtcd macro layer only:
 * av1_apply_temporal_filter / av1_highbd_apply_temporal_filter are #defined to
 * a recorder that stores (subblock_mvs, subblock_mses, pred) per
 * (block, frame) and then calls the reference's own av1_apply_temporal_filter_c.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "config/aom_config.h"
#include "config/aom_dsp_rtcd.h"
#include "config/av1_rtcd.h"
#include "config/aom_scale_rtcd.h"

#include "av1/encoder/encoder.h"
#include "av1/encoder/encoder_utils.h"
#include "av1/encoder/extend.h"
#include "av1/encoder/lookahead.h"

#define TFREF_API __attribute__((visibility("default")))

/* ---- recorder hook ------------------------------------------------------ */
typedef struct {
  int16_t *mvs;    /* [blocks][frames][4][2] (row, col) */
  int32_t *mses;   /* [blocks][frames][4] */
  uint16_t *pred;  /* [blocks][frames][num_pels] (u8 widened) or NULL */
  uint32_t *accum; /* [blocks][num_pels] final */
  uint16_t *count; /* [blocks][num_pels] final */
  int num_frames, num_pels, mb_cols, is_hbd;
  int cur_frame; /* frame index being processed (tracked by the hook) */
  int last_block;
  int filter_frame_idx;
} tfref_rec_t;
static tfref_rec_t g_rec;
static int g_rec_on = 0;
static double g_q = 0.0;

static void tfref_apply_hook(const YV12_BUFFER_CONFIG *frame_to_filter,
                             const MACROBLOCKD *mbd, const BLOCK_SIZE block_size,
                             const int mb_row, const int mb_col,
                             const int num_planes, const double *noise_levels,
                             const MV *subblock_mvs, const int *subblock_mses,
                             const int q_factor, const int filter_strength,
                             const uint8_t *pred, uint32_t *accum,
                             uint16_t *count);

/* whatever the rtcd header bound these names to (_c, or _avx2 in the libtf_ref_avx2.so flavour) */
typedef void (*tfref_apply_fn)(const YV12_BUFFER_CONFIG *, const MACROBLOCKD *, const BLOCK_SIZE,
                               const int, const int, const int, const double *, const MV *,
                               const int *, const int, const int, const uint8_t *, uint32_t *,
                               uint16_t *);
static const tfref_apply_fn tfref_apply_lbd = av1_apply_temporal_filter;
static const tfref_apply_fn tfref_apply_hbd = av1_highbd_apply_temporal_filter;

#undef av1_apply_temporal_filter
#define av1_apply_temporal_filter tfref_apply_hook
#undef av1_highbd_apply_temporal_filter
#define av1_highbd_apply_temporal_filter tfref_apply_hook

#include "av1/encoder/temporal_filter.c"

static void tfref_apply_hook(const YV12_BUFFER_CONFIG *frame_to_filter,
                             const MACROBLOCKD *mbd, const BLOCK_SIZE block_size,
                             const int mb_row, const int mb_col,
                             const int num_planes, const double *noise_levels,
                             const MV *subblock_mvs, const int *subblock_mses,
                             const int q_factor, const int filter_strength,
                             const uint8_t *pred, uint32_t *accum,
                             uint16_t *count) {
  if (g_rec_on) {
    const int blk = mb_row * g_rec.mb_cols + mb_col;
    if (blk != g_rec.last_block) {
      g_rec.last_block = blk;
      g_rec.cur_frame = 0;
    }
    if (g_rec.cur_frame == g_rec.filter_frame_idx) g_rec.cur_frame++;
    const int f = g_rec.cur_frame++;
    const size_t bf = (size_t)blk * g_rec.num_frames + f;
    if (g_rec.mvs) {
      for (int i = 0; i < 4; i++) {
        g_rec.mvs[(bf * 4 + i) * 2 + 0] = subblock_mvs[i].row;
        g_rec.mvs[(bf * 4 + i) * 2 + 1] = subblock_mvs[i].col;
      }
    }
    if (g_rec.mses)
      for (int i = 0; i < 4; i++) g_rec.mses[bf * 4 + i] = subblock_mses[i];
    if (g_rec.pred) {
      uint16_t *dst = g_rec.pred + bf * g_rec.num_pels;
      if (g_rec.is_hbd) {
        memcpy(dst, CONVERT_TO_SHORTPTR(pred), g_rec.num_pels * 2);
      } else {
        for (int i = 0; i < g_rec.num_pels; i++) dst[i] = pred[i];
      }
    }
  }
  ((frame_to_filter->flags & YV12_FLAG_HIGHBITDEPTH) ? tfref_apply_hbd : tfref_apply_lbd)(
      frame_to_filter, mbd, block_size, mb_row, mb_col, num_planes, noise_levels, subblock_mvs,
      subblock_mses, q_factor, filter_strength, pred, accum, count);
}

/* ---- symbols the dropped control-plane would have provided -------------- */
double av1_convert_qindex_to_q(int qindex, aom_bit_depth_t bit_depth) {
  (void)qindex;
  (void)bit_depth;
  return g_q;
}
void aom_internal_error(struct aom_internal_error_info *info,
                        aom_codec_err_t error, const char *fmt, ...) {
  (void)info;
  (void)error;
  (void)fmt;
  abort();
}

/* ---- public harness API -------------------------------------------------- */
typedef struct {
  int width, height; /* luma crop size */
  int ss_x, ss_y, monochrome;
  int bit_depth, use_hbd;
  int border; /* oxcf.border_in_pixels */
  int num_frames, filter_frame_idx;
  double noise_levels[3];
  int q_factor;
  int filter_strength; /* FINAL strength (policy at :813-842 bypassed by
                          arnr_strength=filter_strength, content=default,
                          update_type=ARF) */
  int force_integer_mv, allow_hp;
  int subpel_method;       /* 0 TREE, 1 PRUNED, 2 PRUNED_MORE */
  int subpel_iters_per_step;
  int prune_mesh_level;    /* PRUNE_MESH_SEARCH_{DISABLED,LVL_1,LVL_2} */
  int mesh[4][2];          /* {range, interval} */
  int use_downsampled_sad;
  int compute_frame_diff;
} tfref_cfg;

/* A frame lives inside a lookahead_entry, as in the encoder (lookahead.h:33-39), so the
 * CONFIG_TF_GPU seam can recover display_idx from the YV12 pointer. */
typedef struct {
  struct lookahead_entry entry;
} tfref_frame;
#define buf entry.img
static int g_display_idx = 0;

static int align_pow2(int v, int n) { return (v + (1 << n) - 1) & ~((1 << n) - 1); }

/* Frame container with the reference's layout (aom_scale/generic/yv12config.c
 * :223-258, aom_calc_y_stride yv12config.h:204): allocation is done by the
 * reference's aom_realloc_frame_buffer itself. */
static int tfref_frame_alloc(tfref_frame *f, const tfref_cfg *c) {
  memset(f, 0, sizeof(*f));
  f->entry.display_idx = g_display_idx++;
  return aom_realloc_frame_buffer(&f->buf, c->width, c->height, c->ss_x, c->ss_y,
                                  c->use_hbd, c->border, 0, NULL, NULL, NULL, 0,
                                  0);
}

/* Fill a frame from planar crop-sized data through the reference's own
 * av1_copy_and_extend_frame (av1/encoder/extend.c:113). */
static void tfref_frame_fill(tfref_frame *f, const tfref_cfg *c,
                             const void *const planes[3]) {
  YV12_BUFFER_CONFIG src;
  memset(&src, 0, sizeof(src));
  const int aw = align_pow2(c->width, 3), ah = align_pow2(c->height, 3);
  const int cw = (c->width + c->ss_x) >> c->ss_x, ch = (c->height + c->ss_y) >> c->ss_y;
  src.y_crop_width = c->width;
  src.y_crop_height = c->height;
  src.y_width = aw;
  src.y_height = ah;
  src.uv_crop_width = cw;
  src.uv_crop_height = ch;
  src.uv_width = aw >> c->ss_x;
  src.uv_height = ah >> c->ss_y;
  src.y_stride = c->width;
  src.uv_stride = cw;
  src.subsampling_x = c->ss_x;
  src.subsampling_y = c->ss_y;
  src.monochrome = c->monochrome;
  if (c->use_hbd) {
    src.flags = YV12_FLAG_HIGHBITDEPTH;
    src.y_buffer = CONVERT_TO_BYTEPTR(planes[0]);
    src.u_buffer = planes[1] ? CONVERT_TO_BYTEPTR(planes[1]) : NULL;
    src.v_buffer = planes[2] ? CONVERT_TO_BYTEPTR(planes[2]) : NULL;
  } else {
    src.y_buffer = (uint8_t *)planes[0];
    src.u_buffer = (uint8_t *)planes[1];
    src.v_buffer = (uint8_t *)planes[2];
  }
  f->buf.monochrome = c->monochrome;
  f->entry.display_idx = g_display_idx++; /* new pixels, new id */
  av1_copy_and_extend_frame(&src, &f->buf);
}

typedef struct {
  AV1_COMP *cpi;
  AV1_PRIMARY *ppi;
  SequenceHeader seq;
  struct aom_internal_error_info err;
  tfref_cfg cfg;
  tfref_frame *frames;
  tfref_frame out;
  int num_planes, num_pels, mb_rows, mb_cols;
  const YV12_BUFFER_CONFIG *la_frames[32]; /* seam tests: the window inside a real lookahead */
  int use_lookahead;
} tfref_ctx;

static void set_fn_ptrs(AV1_PRIMARY *ppi, int use_hbd, int bd) {
  aom_variance_fn_ptr_t *p32 = &ppi->fn_ptr[BLOCK_32X32];
  aom_variance_fn_ptr_t *p16 = &ppi->fn_ptr[BLOCK_16X16];
  if (!use_hbd) {
    /* av1/encoder/encoder.c:1065-1078,1204,1208 */
    p32->sdf = aom_sad32x32; p32->vf = aom_variance32x32;
    p32->svf = aom_sub_pixel_variance32x32; p32->sdx4df = aom_sad32x32x4d;
    p32->sdx3df = aom_sad32x32x3d;
    p32->sdsf = aom_sad_skip_32x32; p32->sdsx4df = aom_sad_skip_32x32x4d;
    p16->sdf = aom_sad16x16; p16->vf = aom_variance16x16;
    p16->svf = aom_sub_pixel_variance16x16; p16->sdx4df = aom_sad16x16x4d;
    p16->sdx3df = aom_sad16x16x3d;
    p16->sdsf = aom_sad_skip_16x16; p16->sdsx4df = aom_sad_skip_16x16x4d;
    return;
  }
  /* av1/encoder/encoder_utils.h:140-150,415-422 (highbd_set_var_fns) */
#define SETHBD(BD)                                                          \
  p32->sdf = aom_highbd_sad32x32_bits##BD;                                  \
  p32->vf = aom_highbd_##BD##_variance32x32;                                \
  p32->svf = aom_highbd_##BD##_sub_pixel_variance32x32;                     \
  p32->sdx4df = aom_highbd_sad32x32x4d_bits##BD;                            \
  p32->sdx3df = aom_highbd_sad32x32x3d_bits##BD;                            \
  p32->sdsf = aom_highbd_sad_skip_32x32_bits##BD;                           \
  p32->sdsx4df = aom_highbd_sad_skip_32x32x4d_bits##BD;                     \
  p16->sdf = aom_highbd_sad16x16_bits##BD;                                  \
  p16->vf = aom_highbd_##BD##_variance16x16;                                \
  p16->svf = aom_highbd_##BD##_sub_pixel_variance16x16;                     \
  p16->sdx4df = aom_highbd_sad16x16x4d_bits##BD;                            \
  p16->sdx3df = aom_highbd_sad16x16x3d_bits##BD;                            \
  p16->sdsf = aom_highbd_sad_skip_16x16_bits##BD;                           \
  p16->sdsx4df = aom_highbd_sad_skip_16x16x4d_bits##BD;
  if (bd == 8) { SETHBD(8) } else if (bd == 10) { SETHBD(10) } else { SETHBD(12) }
#undef SETHBD
}

TFREF_API void *tfref_create(const tfref_cfg *cfg) {
  tfref_ctx *t = (tfref_ctx *)calloc(1, sizeof(*t));
  t->cfg = *cfg;
  AV1_COMP *cpi = (AV1_COMP *)calloc(1, sizeof(AV1_COMP));
  AV1_PRIMARY *ppi = (AV1_PRIMARY *)calloc(1, sizeof(AV1_PRIMARY));
  t->cpi = cpi;
  t->ppi = ppi;
  cpi->ppi = ppi;
  AV1_COMMON *cm = &cpi->common;
  cm->seq_params = &t->seq;
  cm->error = &t->err;
  t->seq.bit_depth = (aom_bit_depth_t)cfg->bit_depth;
  t->seq.use_highbitdepth = (uint8_t)cfg->use_hbd;
  t->seq.subsampling_x = cfg->ss_x;
  t->seq.subsampling_y = cfg->ss_y;
  t->seq.monochrome = (uint8_t)cfg->monochrome;
  ppi->seq_params = t->seq;
  cm->width = cfg->width;
  cm->height = cfg->height;
  /* av1/common/alloccommon.c (enc_set_mb_mi): mi units of 4 px over the
   * 8-aligned frame size. */
  cm->mi_params.mi_cols = align_pow2(cfg->width, 3) >> MI_SIZE_LOG2;
  cm->mi_params.mi_rows = align_pow2(cfg->height, 3) >> MI_SIZE_LOG2;
  cm->features.cur_frame_force_integer_mv = cfg->force_integer_mv;
  cm->features.allow_high_precision_mv = cfg->allow_hp;

  cpi->oxcf.border_in_pixels = cfg->border;
  cpi->oxcf.algo_cfg.arnr_strength = cfg->filter_strength;
  cpi->oxcf.tune_cfg.content = AOM_CONTENT_DEFAULT;
  cpi->oxcf.kf_cfg.enable_keyframe_filtering = 0;
  cpi->gf_frame_index = 0;
  ppi->gf_group.update_type[0] = ARF_UPDATE;
  ppi->gf_group.frame_type[0] = INTER_FRAME;
  g_q = (double)cfg->q_factor;

  MV_SPEED_FEATURES *mv_sf = &cpi->sf.mv_sf;
  mv_sf->search_method = NSTEP;
  mv_sf->use_bsize_dependent_search_method = 0;
  mv_sf->use_downsampled_sad = cfg->use_downsampled_sad;
  for (int i = 0; i < 4; i++) {
    mv_sf->mesh_patterns[i].range = cfg->mesh[i][0];
    mv_sf->mesh_patterns[i].interval = cfg->mesh[i][1];
  }
  mv_sf->prune_mesh_search = (PRUNE_MESH_SEARCH_LEVEL)cfg->prune_mesh_level;
  mv_sf->subpel_force_stop = EIGHTH_PEL;
  mv_sf->subpel_iters_per_step = cfg->subpel_iters_per_step;
  mv_sf->use_accurate_subpel_search = USE_8_TAPS;
  mv_sf->use_fullpel_costlist = 0;
  mv_sf->subpel_search_method = cfg->subpel_method == 0   ? SUBPEL_TREE
                                : cfg->subpel_method == 1 ? SUBPEL_TREE_PRUNED
                                                          : SUBPEL_TREE_PRUNED_MORE;
  /* av1/encoder/speed_features.c:2150-2170 */
  cpi->mv_search_params.find_fractional_mv_step =
      cfg->subpel_method == 0   ? av1_find_best_sub_pixel_tree
      : cfg->subpel_method == 1 ? av1_find_best_sub_pixel_tree_pruned
                                : av1_find_best_sub_pixel_tree_pruned_more;
  set_fn_ptrs(ppi, cfg->use_hbd, cfg->bit_depth);

  t->num_planes = cfg->monochrome ? 1 : 3;
  t->num_pels = 1024;
  if (!cfg->monochrome) t->num_pels += 2 * (1024 >> (cfg->ss_x + cfg->ss_y));
  t->mb_rows = (cfg->height + 31) / 32;
  t->mb_cols = (cfg->width + 31) / 32;

  t->frames = (tfref_frame *)calloc(cfg->num_frames, sizeof(tfref_frame));
  for (int i = 0; i < cfg->num_frames; i++) {
    if (tfref_frame_alloc(&t->frames[i], cfg)) return NULL;
  }
  if (tfref_frame_alloc(&t->out, cfg)) return NULL;
  return t;
}

/* cm->mi_params and cm->width / cm->height where the coded size differs from the crop size (superres / resize);
 * 0 keeps the value tfref_create derived from the crop size.  Call before tfref_run.  A setter rather than tfref_cfg
 * fields, so that the layout of tfref_cfg stays what existing callers were built against. */
TFREF_API void tfref_set_coded(void *h, int mi_rows, int mi_cols, int cm_width, int cm_height) {
  AV1_COMMON *cm = &((tfref_ctx *)h)->cpi->common;
  if (mi_rows > 0) cm->mi_params.mi_rows = mi_rows;
  if (mi_cols > 0) cm->mi_params.mi_cols = mi_cols;
  if (cm_width > 0) cm->width = cm_width;
  if (cm_height > 0) cm->height = cm_height;
}

TFREF_API void tfref_set_frame(void *h, int idx, const void *y, const void *u,
                               const void *v) {
  tfref_ctx *t = (tfref_ctx *)h;
  const void *planes[3] = { y, u, v };
  tfref_frame_fill(&t->frames[idx], &t->cfg, planes);
}

TFREF_API void tfref_frame_info(void *h, int *y_stride, int *uv_stride,
                                int *border, int *aligned_w, int *aligned_h) {
  tfref_ctx *t = (tfref_ctx *)h;
  const YV12_BUFFER_CONFIG *b = &t->frames[0].buf;
  *y_stride = b->y_stride;
  *uv_stride = b->uv_stride;
  *border = b->border;
  *aligned_w = b->y_width;
  *aligned_h = b->y_height;
}

/* Copies a whole plane allocation (with borders) of input frame idx (or the
 * output when idx < 0) into dst as u16: rows = plane_h + 2*border_h, row
 * length = stride. Returns stride. */
TFREF_API int tfref_get_plane_with_border(void *h, int idx, int plane,
                                          uint16_t *dst, int *rows) {
  tfref_ctx *t = (tfref_ctx *)h;
  const YV12_BUFFER_CONFIG *b = idx < 0 ? &t->out.buf : &t->frames[idx].buf;
  const int is_uv = plane > 0;
  const int stride = b->strides[is_uv];
  const int bh = is_uv ? (b->border >> t->cfg.ss_y) : b->border;
  const int bw = is_uv ? (b->border >> t->cfg.ss_x) : b->border;
  const int ph = b->heights[is_uv] + 2 * bh;
  *rows = ph;
  const uint8_t *p8 = b->buffers[plane];
  if (t->cfg.use_hbd) {
    const uint16_t *p = CONVERT_TO_SHORTPTR(p8) - bh * stride - bw;
    memcpy(dst, p, (size_t)ph * stride * 2);
  } else {
    const uint8_t *p = p8 - bh * stride - bw;
    for (size_t i = 0; i < (size_t)ph * stride; i++) dst[i] = p[i];
  }
  return stride;
}

/* Runs the reference filter over block rows [row_begin,row_end).  Optional
 * recorders may be NULL.  out_{y,u,v} receive mb_rows*32 x mb_cols*32 (luma)
 * samples as u16 (full blocks, temporal_filter.c:740-777). */
static void tfref_setup_tf_ctx(tfref_ctx *t) {
  AV1_COMP *cpi = t->cpi;
  const tfref_cfg *c = &t->cfg;
  TemporalFilterCtx *tf_ctx = &cpi->tf_ctx;
  for (int i = 0; i < c->num_frames; i++)
    tf_ctx->frames[i] = (YV12_BUFFER_CONFIG *)(t->use_lookahead ? t->la_frames[i] : &t->frames[i].buf);
  tf_ctx->num_frames = c->num_frames;
  tf_ctx->filter_frame_idx = c->filter_frame_idx;
  tf_ctx->output_frame = &t->out.buf;
  tf_ctx->compute_frame_diff = c->compute_frame_diff;
  for (int i = 0; i < 3; i++) tf_ctx->noise_levels[i] = c->noise_levels[i];
  tf_ctx->num_pels = t->num_pels;
  tf_ctx->mb_rows = t->mb_rows;
  tf_ctx->mb_cols = t->mb_cols;
  tf_ctx->is_highbitdepth = c->use_hbd;
  tf_ctx->q_factor = c->q_factor;
  av1_setup_scale_factors_for_frame(&tf_ctx->sf, c->width, c->height, c->width,
                                    c->height);
}

#if CONFIG_TF_GPU
/* The reference-side CONFIG_TF_GPU seam (integration/tf_gpu_seam.patch), driven hunk by hunk: the
 * exact code a maintainer adds, filling tf_gpu_params / tf_gpu_frame from AV1_COMP and calling
 * libtf_gpu.so. */
/* The patch's replacement for the noise-estimation loop of tf_setup_filtering_buffer(). */
TFREF_API void tfref_gpu_noise_levels(void *h, int idx, double *noise_levels) {
  tfref_ctx *t = (tfref_ctx *)h;
  tf_gpu_noise_levels(t->cpi, &t->frames[idx].entry, noise_levels);
}

/* av1_tf_gpu_estimate_noise() as the key-frame gate (encode_strategy.c:746-750, in_lookahead = 1) and the
 * ALLINTRA noise synthesis (encoder.c:4038-4051, in_lookahead = 0, edge threshold 16) call it. */
TFREF_API double tfref_gpu_estimate_noise(void *h, int idx, int in_lookahead, int plane, int edge_thresh) {
  tfref_ctx *t = (tfref_ctx *)h;
  return av1_tf_gpu_estimate_noise(t->cpi, &t->frames[idx].buf, in_lookahead, plane, t->cfg.bit_depth,
                                   edge_thresh);
}

/* av1_temporal_filter()'s branch: the synchronous call. */
TFREF_API void tfref_run_gpu_seam(void *h, int64_t *diff_sum_sse) {
  tfref_ctx *t = (tfref_ctx *)h;
  tfref_setup_tf_ctx(t);
  FRAME_DIFF fd = { 0, 0 };
  tf_gpu_do_filtering(t->cpi, t->cfg.compute_frame_diff ? &fd : NULL);
  if (diff_sum_sse) {
    diff_sum_sse[0] = fd.sum;
    diff_sum_sse[1] = fd.sse;
  }
}

/* av1_tf_info_filtering()'s branch: `copies` submits of the same window back to back (as the KF and ARF
 * windows of a GOP), waited for together; the output comes back with aom_extend_frame_borders() already
 * applied on the device.  Every copy writes t->out; diff_sum_sse receives the last one's FRAME_DIFF and
 * *all_equal whether every copy reported the same. */
TFREF_API void tfref_run_gpu_seam_async(void *h, int copies, int64_t *diff_sum_sse, int *all_equal) {
  tfref_ctx *t = (tfref_ctx *)h;
  tfref_setup_tf_ctx(t);
  uint64_t ticket[8];
  int64_t diff[8][2];
  if (copies > 8) copies = 8;
  for (int i = 0; i < copies; i++) ticket[i] = tf_gpu_submit_filtering(t->cpi, diff[i]);
  FRAME_DIFF fd = { 0, 0 };
  *all_equal = 1;
  for (int i = 0; i < copies; i++) {
    tf_gpu_wait_filtering(t->cpi, ticket[i], diff[i], &fd);
    if (diff[i][0] != diff[0][0] || diff[i][1] != diff[0][1]) *all_equal = 0;
  }
  diff_sum_sse[0] = fd.sum;
  diff_sum_sse[1] = fd.sse;
}

/* The av1_receive_raw_frame() hunk: a real lookahead (av1_lookahead_init / av1_lookahead_push), every
 * pushed frame uploaded by av1_tf_gpu_lookahead_push(); afterwards the window's frames[] point at the
 * lookahead entries, as tf_setup_filtering_buffer() leaves them. */
TFREF_API int tfref_gpu_push_window(void *h) {
  tfref_ctx *t = (tfref_ctx *)h;
  const tfref_cfg *c = &t->cfg;
  AV1_COMP *cpi = t->cpi;
  if (!t->ppi->lookahead)
    t->ppi->lookahead = av1_lookahead_init(c->width, c->height, c->ss_x, c->ss_y, c->use_hbd,
                                           c->num_frames, c->border, 0, 0, false, 0);
  if (!t->ppi->lookahead) return -1;
  cpi->compressor_stage = ENCODE_STAGE;
  cpi->oxcf.pass = AOM_RC_ONE_PASS;
  t->ppi->tf_info.is_temporal_filter_on = 1;
  for (int i = 0; i < c->num_frames; i++) {
    if (av1_lookahead_push(t->ppi->lookahead, &t->frames[i].buf, i, i + 1, c->use_hbd, 0, 0)) return -2;
    av1_tf_gpu_lookahead_push(cpi);
  }
  for (int i = 0; i < c->num_frames; i++) {
    struct lookahead_entry *e = av1_lookahead_peek(t->ppi->lookahead, i, ENCODE_STAGE);
    if (!e) return -3;
    t->la_frames[i] = &e->img;
  }
  t->use_lookahead = 1;
  return 0;
}

/* kernel launches of the last library call on the seam's context (uploads show up as border kernels) */
TFREF_API int tfref_gpu_last_launches(void *h) {
  tfref_ctx *t = (tfref_ctx *)h;
  int n = -1;
  if (t->ppi->tf_info.gpu) tf_gpu_last_stats(t->ppi->tf_info.gpu, &n, NULL);
  return n;
}
TFREF_API int tfref_gpu_num_pinned(void *h) { return ((tfref_ctx *)h)->ppi->tf_info.gpu_num_pinned; }
TFREF_API int tfref_gpu_has_context(void *h) { return ((tfref_ctx *)h)->ppi->tf_info.gpu != NULL; }
/* av1_tf_info_free()'s hunk: the context dies with the TEMPORAL_FILTER_INFO */
TFREF_API void tfref_gpu_release(void *h) {
  tfref_ctx *t = (tfref_ctx *)h;
  const int on = t->ppi->tf_info.is_temporal_filter_on;
  t->ppi->tf_info.is_temporal_filter_on = 0; /* the harness owns no tf_buf[] */
  av1_tf_info_free(&t->ppi->tf_info);
  t->ppi->tf_info.is_temporal_filter_on = on;
}
#endif

TFREF_API void tfref_run(void *h, int row_begin, int row_end, int16_t *mvs,
                         int32_t *mses, uint16_t *pred, uint32_t *accum,
                         uint16_t *count, int64_t *diff_sum_sse) {
  tfref_ctx *t = (tfref_ctx *)h;
  AV1_COMP *cpi = t->cpi;
  const tfref_cfg *c = &t->cfg;
  TemporalFilterCtx *tf_ctx = &cpi->tf_ctx;
  tfref_setup_tf_ctx(t);

  ThreadData *td = &cpi->td;
  MACROBLOCKD *mbd = &td->mb.e_mbd;
  /* what tf_setup_filtering_buffer :1138-1142 does */
  mbd->cur_buf = &t->frames[c->filter_frame_idx].buf;
  mbd->bd = c->bit_depth;
  for (int p = 0; p < 3; p++) {
    mbd->plane[p].subsampling_x = p ? c->ss_x : 0;
    mbd->plane[p].subsampling_y = p ? c->ss_y : 0;
  }
  mbd->error_info = &t->err;
  tf_alloc_and_reset_data(&td->tf_data, t->num_pels, c->use_hbd);
  tf_setup_macroblockd(mbd, &td->tf_data, &tf_ctx->sf);

  memset(&g_rec, 0, sizeof(g_rec));
  g_rec.mvs = mvs;
  g_rec.mses = mses;
  g_rec.pred = pred;
  g_rec.num_frames = c->num_frames;
  g_rec.num_pels = t->num_pels;
  g_rec.mb_cols = t->mb_cols;
  g_rec.is_hbd = c->use_hbd;
  g_rec.filter_frame_idx = c->filter_frame_idx;
  g_rec.last_block = -1;
  g_rec_on = 1;
  (void)accum;
  (void)count;
  for (int r = row_begin; r < row_end; r++) av1_tf_do_filtering_row(cpi, td, r);
  g_rec_on = 0;
  if (diff_sum_sse) {
    diff_sum_sse[0] = td->tf_data.diff.sum;
    diff_sum_sse[1] = td->tf_data.diff.sse;
  }
  tf_dealloc_data(&td->tf_data, c->use_hbd);
}

#pragma push_macro("buf")
#undef buf /* struct buf_2d has a member of that name */
/* av1_full_pixel_search() (mcomp.c:1693-1832) on one block, configured exactly as tf_motion_search()
 * configures it (temporal_filter.c:104-160: NSTEP sites for the frame stride, step_param from the frame size,
 * L1 MV cost class, mesh search on, LVL_1 pruning by q) -- the search first_pass_motion_search()
 * (firstpass.c:261-300) and TPL's motion_estimation() (tpl_model.c:285) also run per block.  The block is the
 * bsize x bsize (16 or 32) block of frame src_idx at luma position (x, y), searched in frame ref_idx from the
 * full-pel start MV; MV limits from av1_set_mv_{row,col}_limits for that block.  out = {row, col, var}. */
TFREF_API void tfref_full_pixel_search(void *h, int src_idx, int ref_idx, int bsize, int x, int y,
                                       int start_row, int start_col, int *out) {
  tfref_ctx *t = (tfref_ctx *)h;
  AV1_COMP *cpi = t->cpi;
  const tfref_cfg *c = &t->cfg;
  tfref_setup_tf_ctx(t);
  ThreadData *td = &cpi->td;
  MACROBLOCK *mb = &td->mb;
  MACROBLOCKD *mbd = &mb->e_mbd;
  mbd->cur_buf = &t->frames[src_idx].entry.img;
  mbd->bd = c->bit_depth;
  for (int p = 0; p < 3; p++) {
    mbd->plane[p].subsampling_x = p ? c->ss_x : 0;
    mbd->plane[p].subsampling_y = p ? c->ss_y : 0;
  }
  mbd->error_info = &t->err;
  tf_alloc_and_reset_data(&td->tf_data, t->num_pels, c->use_hbd);
  tf_setup_macroblockd(mbd, &td->tf_data, &cpi->tf_ctx.sf);
  const BLOCK_SIZE block_size = bsize == 32 ? BLOCK_32X32 : BLOCK_16X16;
  const YV12_BUFFER_CONFIG *frame_to_filter = &t->frames[src_idx].entry.img;
  const YV12_BUFFER_CONFIG *ref_frame = &t->frames[ref_idx].entry.img;
  const int y_stride = frame_to_filter->y_stride;
  const int y_offset = y * y_stride + x;
  av1_set_mv_row_limits(&cpi->common.mi_params, &mb->mv_limits, y >> MI_SIZE_LOG2, bsize >> MI_SIZE_LOG2,
                        cpi->oxcf.border_in_pixels);
  av1_set_mv_col_limits(&cpi->common.mi_params, &mb->mv_limits, x >> MI_SIZE_LOG2, bsize >> MI_SIZE_LOG2,
                        cpi->oxcf.border_in_pixels);
  /* from here on: tf_motion_search() :94-160, verbatim in meaning */
  const int min_frame_size = AOMMIN(cpi->common.width, cpi->common.height);
  const struct buf_2d ori_src_buf = mb->plane[0].src;
  const struct buf_2d ori_pre_buf = mbd->plane[0].pre[0];
  FULLPEL_MOTION_SEARCH_PARAMS full_ms_params;
  const SEARCH_METHODS search_method = NSTEP;
  const search_site_config *search_site_cfg =
      av1_get_search_site_config(mb->search_site_cfg_buf, &cpi->mv_search_params, search_method, y_stride);
  const int step_param =
      av1_init_search_range(AOMMAX(frame_to_filter->y_crop_width, frame_to_filter->y_crop_height));
  const MV_COST_TYPE mv_cost_type =
      min_frame_size >= 720 ? MV_COST_L1_HDRES
                            : (min_frame_size >= 480 ? MV_COST_L1_MIDRES : MV_COST_L1_LOWRES);
  FULLPEL_MV start_mv = { (int16_t)start_row, (int16_t)start_col };
  const MV baseline_mv = kZeroMv;
  mb->plane[0].src.buf = frame_to_filter->y_buffer + y_offset;
  mb->plane[0].src.stride = y_stride;
  mbd->plane[0].pre[0].buf = ref_frame->y_buffer + y_offset;
  mbd->plane[0].pre[0].stride = y_stride;
  int cost_list[5];
  int_mv best_mv;
  const int q = av1_get_q(cpi);
  av1_make_default_fullpel_ms_params(&full_ms_params, cpi, mb, block_size, &baseline_mv, search_site_cfg,
                                     /*fine_search_interval=*/0);
  av1_set_mv_search_method(&full_ms_params, search_site_cfg, search_method);
  full_ms_params.run_mesh_search = 1;
  full_ms_params.mv_cost_params.mv_cost_type = mv_cost_type;
  if (cpi->sf.mv_sf.prune_mesh_search == PRUNE_MESH_SEARCH_LVL_1) {
    full_ms_params.prune_mesh_search = (q <= 20) ? 0 : 1;
    full_ms_params.mesh_search_mv_diff_threshold = 2;
  }
  const int var = av1_full_pixel_search(start_mv, &full_ms_params, step_param, cond_cost_list(cpi, cost_list),
                                        &best_mv.as_fullmv, NULL);
  out[0] = best_mv.as_fullmv.row;
  out[1] = best_mv.as_fullmv.col;
  out[2] = var;
  mb->plane[0].src = ori_src_buf;
  mbd->plane[0].pre[0] = ori_pre_buf;
  tf_dealloc_data(&td->tf_data, c->use_hbd);
}

#pragma pop_macro("buf")

/* Output plane (full blocks region) as u16. w,h = number of samples copied. */
TFREF_API void tfref_get_output(void *h, int plane, uint16_t *dst, int w, int hgt) {
  tfref_ctx *t = (tfref_ctx *)h;
  const YV12_BUFFER_CONFIG *b = &t->out.buf;
  const int is_uv = plane > 0;
  const int stride = b->strides[is_uv];
  for (int y = 0; y < hgt; y++) {
    for (int x = 0; x < w; x++) {
      dst[(size_t)y * w + x] =
          t->cfg.use_hbd ? CONVERT_TO_SHORTPTR(b->buffers[plane])[y * stride + x]
                         : b->buffers[plane][y * stride + x];
    }
  }
}

TFREF_API double tfref_estimate_noise(void *h, int idx, int plane) {
  tfref_ctx *t = (tfref_ctx *)h;
  return av1_estimate_noise_from_single_plane(&t->frames[idx].buf, plane,
                                              t->cfg.bit_depth,
                                              NOISE_ESTIMATION_EDGE_THRESHOLD);
}

TFREF_API void tfref_extend_output_borders(void *h) {
  tfref_ctx *t = (tfref_ctx *)h;
  aom_extend_frame_borders_c(&t->out.buf, t->num_planes);
}

TFREF_API void tfref_destroy(void *h) {
  tfref_ctx *t = (tfref_ctx *)h;
  if (!t) return;
#if CONFIG_TF_GPU
  tfref_gpu_release(h);
  if (t->ppi->lookahead) av1_lookahead_destroy(t->ppi->lookahead);
#endif
  for (int i = 0; i < t->cfg.num_frames; i++) aom_free_frame_buffer(&t->frames[i].buf);
  aom_free_frame_buffer(&t->out.buf);
  free(t->frames);
  free(t->cpi);
  free(t->ppi);
  free(t);
}

/* ---- unit-level entry points --------------------------------------------- */

/* The reference's av1_apply_temporal_filter_c on caller-supplied block data,
 * the exact call test/temporal_filter_test.cc:210-221 makes.  src planes are
 * tightly packed W x H; pred is planar [Y][U][V]. */
TFREF_API void tfref_apply_block(int width, int height, int ss_x, int ss_y,
                                 int num_planes, int bd, int use_hbd,
                                 const void *src_y, const void *src_u,
                                 const void *src_v, int y_stride, int uv_stride,
                                 int mb_row, int mb_col,
                                 const double *noise_levels, const int16_t *mvs,
                                 const int *mses, int q_factor, int strength,
                                 const void *pred, uint32_t *accum,
                                 uint16_t *count) {
  YV12_BUFFER_CONFIG f;
  memset(&f, 0, sizeof(f));
  f.y_crop_width = width;
  f.y_crop_height = height;
  f.y_stride = y_stride;
  f.uv_stride = uv_stride;
  f.flags = use_hbd ? YV12_FLAG_HIGHBITDEPTH : 0;
  f.y_buffer = use_hbd ? CONVERT_TO_BYTEPTR(src_y) : (uint8_t *)src_y;
  f.u_buffer = use_hbd ? CONVERT_TO_BYTEPTR(src_u) : (uint8_t *)src_u;
  f.v_buffer = use_hbd ? CONVERT_TO_BYTEPTR(src_v) : (uint8_t *)src_v;
  MACROBLOCKD *mbd = (MACROBLOCKD *)calloc(1, sizeof(MACROBLOCKD));
  mbd->bd = bd;
  for (int p = 0; p < 3; p++) {
    mbd->plane[p].subsampling_x = p ? ss_x : 0;
    mbd->plane[p].subsampling_y = p ? ss_y : 0;
  }
  MV m[4];
  for (int i = 0; i < 4; i++) { m[i].row = mvs[2 * i]; m[i].col = mvs[2 * i + 1]; }
  const uint8_t *pred8 = use_hbd ? CONVERT_TO_BYTEPTR(pred) : (const uint8_t *)pred;
  av1_apply_temporal_filter_c(&f, mbd, BLOCK_32X32, mb_row, mb_col, num_planes,
                              noise_levels, m, mses, q_factor, strength, pred8,
                              accum, count);
  free(mbd);
}

/* OD_DIVU (aom_dsp/odintrin.h:30-42) probes: single value, and an exhaustive
 * comparison with plain integer division over d in [dmin,dmax], x in [0,xmax]. */
TFREF_API unsigned tfref_od_divu(unsigned x, unsigned d) { return OD_DIVU(x, d); }
TFREF_API long long tfref_od_divu_mismatches(unsigned dmin, unsigned dmax, unsigned xmax) {
  long long bad = 0;
  for (unsigned d = dmin; d <= dmax; d++)
    for (unsigned x = 0; x <= xmax; x++) bad += (OD_DIVU(x, d) != x / d);
  return bad;
}
