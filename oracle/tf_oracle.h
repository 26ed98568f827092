/*
 * TEST INFRASTRUCTURE -- CPU restatement ("oracle") of the reference's
 * temporal-filter hot path (av1/encoder/temporal_filter.c and the mcomp /
 * convolve / sad / variance subset it calls).  Only tests/, bench.py's
 * cpu_baseline leg and __graft_entry__.smoke() may load it; the product
 * (libtf_gpu.so) never links, loads or calls anything in oracle/.
 *
 * Parity status: PINNED -- checked bit-for-bit against the unmodified
 * reference compiled into oracle/_ref/libtf_ref.so (tests/test_oracle_vs_ref.py)
 * and against fixtures generated from it (tests/golden/).
 */
#ifndef TF_ORACLE_H_
#define TF_ORACLE_H_
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct {
  int width, height; /* luma crop size */
  int ss_x, ss_y, monochrome;
  int bit_depth, use_hbd;
  int border; /* oxcf.border_in_pixels (enters the MV limits only) */
  int num_frames, filter_frame_idx;
  double noise_levels[3];
  int q_factor;
  int filter_strength; /* final strength, after temporal_filter.c:813-842 */
  int force_integer_mv, allow_hp;
  int subpel_method; /* 0 TREE, 1 PRUNED, 2 PRUNED_MORE */
  int subpel_iters_per_step;
  int prune_mesh_level; /* 0 off, 1 LVL_1 (q-dependent, thr 2), 2 LVL_2 (thr 4) */
  int mesh[4][2];       /* {range, interval} */
  int use_downsampled_sad;
  int compute_frame_diff;
} tfo_params;

typedef struct tfo_ctx tfo_ctx;

tfo_ctx *tfo_create(const tfo_params *p);
/* cm->mi_params.mi_rows / mi_cols (4-px units; the MV limits, mcomp.h:216-240) and cm->width / cm->height (the coded
 * size: MV cost class and ref_mv reset threshold, temporal_filter.c:99-100,119-122,249-250), which differ from the
 * crop size under superres / resize.  0 = derived from the crop size (what tfo_create sets): align8(crop) / 4, and
 * the crop size itself.  Call before any search.  A setter rather than tfo_params fields, so that the layout of
 * tfo_params stays what existing callers were built against. */
void tfo_set_coded(tfo_ctx *c, int mi_rows, int mi_cols, int cm_width, int cm_height);
void tfo_destroy(tfo_ctx *c);
/* planes: crop-sized, tightly packed, u8 (use_hbd=0) or u16 (use_hbd=1) */
void tfo_set_frame(tfo_ctx *c, int idx, const void *y, const void *u, const void *v);
double tfo_estimate_noise(tfo_ctx *c, int idx, int plane);
/* av1_estimate_noise_from_single_plane with an explicit edge_thresh (tfo_estimate_noise passes 50) */
double tfo_estimate_noise_thresh(tfo_ctx *c, int idx, int plane, int edge_thresh);
/* Runs block rows [row_begin,row_end). Recorders may be NULL:
 *  mvs  [blocks][frames][4][2] int16 (row,col); mses [blocks][frames][4] int32;
 *  pred [blocks][frames][num_pels] u16; accum/count [blocks][num_pels]. */
void tfo_run(tfo_ctx *c, int row_begin, int row_end, int16_t *mvs, int32_t *mses,
             uint16_t *pred, uint32_t *accum, uint16_t *count, int64_t *diff_sum_sse);
/* Output plane, full-block region (mb_cols*32>>ss_x by mb_rows*32>>ss_y), as u16 */
void tfo_get_output(tfo_ctx *c, int plane, uint16_t *dst, int w, int h);
/* Whole padded input plane (idx>=0) as u16: returns stride, *rows, *border_px */
int tfo_get_plane_with_border(tfo_ctx *c, int idx, int plane, uint16_t *dst, int *rows,
                              int *bw, int *bh);
int tfo_plane_alloc_size(tfo_ctx *c, int plane);
/* aom_extend_frame_borders on the output frame (what the caller runs after the filter) */
void tfo_extend_output_borders(tfo_ctx *c);
/* av1_full_pixel_search as tf_motion_search() configures it, on the bsize x bsize (16 or 32) luma block
 * at (x, y) of frame src_idx against frame ref_idx from full-pel start (start_row, start_col):
 * out = best row, best col, returned variance cost */
void tfo_full_pixel_search(tfo_ctx *c, int src_idx, int ref_idx, int bsize, int x, int y,
                           int start_row, int start_col, int *out);

/* av1_apply_temporal_filter_c on caller supplied block data
 * (the call test/temporal_filter_test.cc:210-221 makes). */
void tfo_apply_block(int width, int height, int ss_x, int ss_y, int num_planes, int bd,
                     int use_hbd, const void *src_y, const void *src_u, const void *src_v,
                     int y_stride, int uv_stride, int mb_row, int mb_col,
                     const double *noise_levels, const int16_t *mvs, const int *mses,
                     int q_factor, int strength, const void *pred, uint32_t *accum,
                     uint16_t *count);

/* primitives, exposed for unit tests (u16 sample buffers) */
unsigned tfo_sad(const uint16_t *a, int as, const uint16_t *b, int bs, int w, int h, int skip,
                 int bd, int use_hbd);
unsigned tfo_variance(const uint16_t *a, int as, const uint16_t *b, int bs, int w, int h,
                      int bd, int use_hbd, unsigned *sse);
unsigned tfo_subpel_variance(const uint16_t *ref, int rs, int xoff, int yoff,
                             const uint16_t *src, int ss, int w, int h, int bd, int use_hbd,
                             unsigned *sse);
void tfo_convolve12(const uint16_t *src, int ss, uint16_t *dst, int ds, int w, int h,
                    int subpel_x, int subpel_y, int bd, int use_hbd);
int tfo_od_divu(unsigned x, unsigned d);

/* Event counters: they only observe, never change a result.  They show that a test input reaches the
 * regime it targets (exact ties, int16 wrap of the 2-D intermediate, clamped predictor samples, ...).
 * One process-wide set; tfo_reset_stats() zeroes it. */
typedef struct {
  int64_t mesh_searches;      /* full_pixel_exhaustive calls that run the mesh (range/interval valid) */
  int64_t diamond_ties;       /* diamond candidates whose sad + cost equals the incumbent (strict < keeps it) */
  int64_t mesh_ties;          /* mesh candidates whose sad + cost equals the incumbent */
  int64_t subpel_ties;        /* sub-pel candidates whose error equals the incumbent */
  int64_t conv_im_overflow;   /* 2-D convolve intermediates outside int16 before the cast */
  int64_t pred_clip_lo;       /* predictor samples clamped to 0 by clip_px */
  int64_t pred_clip_hi;       /* predictor samples clamped to (1 << bd) - 1 by clip_px */
  int64_t mv_on_limit;        /* full-pel MVs (32x32 and 16x16) on a row or column search limit */
  int64_t mv_on_clamp;        /* of those, on a limit set by the +-1023 clamp */
  int64_t ref_mv_resets;      /* block_mse > thresh: ref_mv reset to zero */
  int64_t block_mse_at_thresh; /* block_mse == thresh exactly (the reset's boundary) */
  int64_t sad_peak_groups;    /* 16-sample aligned row groups of a SAD whose every |difference| is (1 << bd) - 1 */
} tfo_stats;
/* Counters of the MV limits, in a struct of their own (tfo_stats keeps its layout); tfo_reset_stats zeroes them too. */
typedef struct {
  int64_t lim_inverted;       /* MV limits with an empty row or column interval (min > max) */
  int64_t start_clamped;      /* search starts moved by the clamp into the limits (diamond and mesh) */
  int64_t lim_border_bound;   /* MV limits with a bound set by the border_in_pixels term (strictly tighter than
                                 the +-8 term and inside the +-1023 clamp) */
} tfo_limit_stats;
void tfo_reset_stats(void);
void tfo_get_stats(tfo_stats *out);
void tfo_get_limit_stats(tfo_limit_stats *out);

#ifdef __cplusplus
}
#endif
#endif
