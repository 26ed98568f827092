/*
 * tf_gpu.h -- C ABI of the B200 temporal filter (libtf_gpu.so).
 *
 * This is the drop-in boundary for the aom-av1-psy encoder's temporal filter
 * (ARNR / ARF denoising).  The reference has no plugin API for this path; the
 * seam is av1_temporal_filter() (av1/encoder/temporal_filter.c:1276): under
 * CONFIG_TF_GPU it calls tf_gpu_filter() after init_tf_ctx() (:1291) instead of
 * tf_alloc_and_reset_data() ... tf_do_filtering(_mt)() (:1296-1311).  See
 * INTEGRATION.md for the patch.  Plain C: POD structs, host pointers and sizes,
 * integer return codes (0 ok, <0 error; never longjmp / exceptions).  There is
 * NO CPU fallback: every entry point fails with TF_GPU_ERR_NO_DEVICE when no
 * CUDA device is usable.
 *
 * Each declaration cites the reference interface it replaces.
 */
#ifndef TF_GPU_H_
#define TF_GPU_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TF_GPU_ABI_VERSION 2
#define TF_GPU_MAX_FRAMES 24 /* reference: arnr_max_frames 15 + adjust 6 = 21 (temporal_filter.c:997,1063-1080) */

enum {
  TF_GPU_OK = 0,
  TF_GPU_ERR_INVALID = -1,   /* bad argument (caller: AOM_CODEC_INVALID_PARAM) */
  TF_GPU_ERR_MEM = -2,       /* device/host allocation failed (caller: AOM_CODEC_MEM_ERROR, cf. temporal_filter.c:1296-1299) */
  TF_GPU_ERR_CUDA = -3,      /* CUDA runtime error (caller: AOM_CODEC_ERROR) */
  TF_GPU_ERR_NO_DEVICE = -4, /* no usable GPU; there is no CPU fallback */
  TF_GPU_ERR_UNSUPPORTED = -5
};

/* Sub-pel search variant = cpi->mv_search_params.find_fractional_mv_step
 * (av1/encoder/speed_features.c:2150-2170, mcomp.c:2844/2929/3065). */
enum { TF_GPU_SUBPEL_TREE = 0, TF_GPU_SUBPEL_TREE_PRUNED = 1, TF_GPU_SUBPEL_TREE_PRUNED_MORE = 2 };
/* PRUNE_MESH_SEARCH_LEVEL (av1/encoder/speed_features.h) */
enum { TF_GPU_PRUNE_MESH_DISABLED = 0, TF_GPU_PRUNE_MESH_LVL_1 = 1, TF_GPU_PRUNE_MESH_LVL_2 = 2 };

typedef struct tf_gpu_ctx tf_gpu_ctx;

typedef struct {
  int device;              /* CUDA device ordinal, -1 = current device */
  int max_cached_frames;   /* device frame-cache slots (0 = default 32) */
  int reserved[6];
} tf_gpu_device_cfg;

/* POD mirror of the YV12_BUFFER_CONFIG fields the temporal filter reads
 * (aom_scale/yv12config.h:43-123).  plane[] point at pixel (0,0) of each plane
 * in HOST memory, already CONVERT_TO_SHORTPTR'd for high bitdepth
 * (aom_ports/mem.h:79-80); strides are in samples.  The pixels outside the
 * crop area must be edge replication, which is what av1_copy_and_extend_frame
 * (av1/encoder/extend.c:113-163) leaves in every lookahead slot; only the crop
 * area is read from the host, borders are rebuilt on the device. */
typedef struct {
  const void *plane[3];
  int stride[2];     /* y_stride, uv_stride (samples) */
  int crop_w[2];     /* y_crop_width, uv_crop_width */
  int crop_h[2];     /* y_crop_height, uv_crop_height */
  int aligned_w[2];  /* y_width, uv_width   (widths[]: 8-aligned luma size >> ss) */
  int aligned_h[2];  /* y_height, uv_height */
  int border;        /* luma border of the host allocation (samples) */
  int ss_x, ss_y;    /* subsampling_x/y */
  int is_hbd;        /* flags & YV12_FLAG_HIGHBITDEPTH */
  uint64_t frame_id; /* lookahead display index (lookahead.h:37): same id => same pixels; 0 = never cache */
} tf_gpu_frame;

/* Everything av1_tf_do_filtering_row (temporal_filter.c:788-939) and
 * tf_motion_search (:87-253) read from AV1_COMP, resolved to plain values. */
typedef struct {
  int num_frames;        /* tf_ctx.num_frames */
  int filter_frame_idx;  /* tf_ctx.filter_frame_idx */
  int num_planes;        /* av1_num_planes(cm): 1 or 3 */
  int bit_depth;         /* seq_params->bit_depth / mbd->bd: 8, 10, 12 */
  double noise_levels[3];/* tf_ctx.noise_levels (temporal_filter.c:1023-1027) */
  int q_factor;          /* av1_get_q(cpi) (:779-786) */
  int filter_strength;   /* FINAL strength after the psy / key-frame overrides (:813-842) */
  int mi_rows, mi_cols;  /* cm->mi_params (4-px units of the 8-aligned frame) */
  int border_in_pixels;  /* oxcf.border_in_pixels (enters av1_set_mv_*_limits, mcomp.h:216-240) */
  int force_integer_mv;  /* cm->features.cur_frame_force_integer_mv */
  int allow_hp;          /* cm->features.allow_high_precision_mv */
  int subpel_method;     /* TF_GPU_SUBPEL_* */
  int subpel_iters_per_step; /* sf.mv_sf.subpel_iters_per_step */
  int prune_mesh_level;  /* sf.mv_sf.prune_mesh_search */
  int mesh_patterns[4][2]; /* sf.mv_sf.mesh_patterns[i].{range,interval} */
  int use_downsampled_sad; /* sf.mv_sf.use_downsampled_sad */
  int compute_frame_diff;  /* frame_diff != NULL (:1283) */
  int out_row_begin, out_row_end; /* slab mode: 32-px block rows [begin,end); 0,0 = all rows */
  /* 1: also run aom_extend_frame_borders (aom_scale/generic/yv12extend.c:221; called right after
   * av1_temporal_filter at temporal_filter.c:1372, encode_strategy.c:822) on the device and return the
   * whole extended allocation of `out` (needs out->border and out->stride to describe it). */
  int extend_output_borders;
  /* cm->width / cm->height: tf_motion_search() picks the MV cost class and the ref_mv reset
   * threshold from AOMMIN(cm->width, cm->height) (temporal_filter.c:99-100,119-122,249-250), which is
   * the CODED size and differs from the source crop size under superres / spatial resize.
   * 0 = use the luma crop size of the frames. */
  int cm_width, cm_height;
  int reserved[5];
} tf_gpu_params;

/* Per-(block, frame) intermediate state for parity tests (what a debug build of
 * the reference would dump from av1_tf_do_filtering_row).  All pointers are
 * optional HOST buffers. */
typedef struct {
  int16_t *subblock_mvs;   /* [blocks][num_frames][4][2] (row,col) 1/8 pel */
  int32_t *subblock_mses;  /* [blocks][num_frames][4] */
  uint16_t *pred;          /* [blocks][num_frames][num_pels] */
  uint32_t *accum;         /* [blocks][num_pels] */
  uint16_t *count;         /* [blocks][num_pels] */
} tf_gpu_dump;

int tf_gpu_abi_version(void);

/* Replaces nothing in the reference (it has no device): context = one CUDA
 * device + stream + frame cache.  Analogue of tf_alloc_and_reset_data
 * (temporal_filter.h:354) hoisted out of the per-call path. */
int tf_gpu_create(tf_gpu_ctx **ctx, const tf_gpu_device_cfg *cfg);
void tf_gpu_destroy(tf_gpu_ctx *ctx);
const char *tf_gpu_last_error(const tf_gpu_ctx *ctx);

/* av1_estimate_noise_from_single_plane (temporal_filter.c:1150-1194), called by
 * tf_setup_filtering_buffer (:1023-1027) and the key-frame gate
 * (encode_strategy.c:746-750).  Uploads (and caches) the frame. */
int tf_gpu_estimate_noise(tf_gpu_ctx *ctx, const tf_gpu_frame *frame, int plane,
                          int bit_depth, int edge_thresh, double *noise_level);

/* The body of av1_temporal_filter (temporal_filter.c:1294-1311): for every
 * 32x32 block, motion search + predictor + weighting against each frame of the
 * window, normalisation into `out`, optional FRAME_DIFF {sum, sse}
 * (temporal_filter.h:83-86).  Synchronous; host buffers are only used during
 * the call.  `out` planes receive full blocks (mb_rows*32 x mb_cols*32 luma
 * samples, as temporal_filter.c:740-777 writes them). */
int tf_gpu_filter(tf_gpu_ctx *ctx, const tf_gpu_params *params,
                  const tf_gpu_frame *frames /*[num_frames]*/, tf_gpu_frame *out,
                  int64_t diff_sum_sse[2] /* nullable */);

/* Same, additionally returning the per-block intermediate state. */
int tf_gpu_filter_dump(tf_gpu_ctx *ctx, const tf_gpu_params *params,
                       const tf_gpu_frame *frames, tf_gpu_frame *out,
                       int64_t diff_sum_sse[2], const tf_gpu_dump *dump);

/* Asynchronous pair for pipelined callers (KF + ARF windows of one GOP are
 * issued back to back by av1_tf_info_filtering, temporal_filter.c:1358-1377):
 * submit enqueues upload + kernels + download on the context's stream and
 * returns a ticket; wait blocks until that ticket's output is in `out`. */
int tf_gpu_submit(tf_gpu_ctx *ctx, const tf_gpu_params *params,
                  const tf_gpu_frame *frames, tf_gpu_frame *out,
                  int64_t diff_sum_sse[2], uint64_t *ticket);
int tf_gpu_wait(tf_gpu_ctx *ctx, uint64_t ticket);

/* Step before / after the path (SURVEY 8f rank 1-2): upload a source frame
 * into the device cache when it enters the lookahead (av1_lookahead_push,
 * lookahead.c:101-163) so that tf_gpu_filter never waits on PCIe; drop it when
 * it leaves.  A cache slot is filled from host memory (tf_gpu_cache_frame,
 * tf_gpu_cache_frame_async, or any call taking tf_gpu_frame) or from device
 * memory (tf_gpu_cache_frame_device); both leave sample-identical slots (crop
 * area plus the replicated device border), so the resident calls cannot tell
 * them apart and one window may mix them. */
int tf_gpu_cache_frame(tf_gpu_ctx *ctx, const tf_gpu_frame *frame);
/* Same without waiting for the copy: the call first waits for the PREVIOUS asynchronous upload of
 * this context, then enqueues this one and returns.  So at most one upload is outstanding and a
 * host buffer may be rewritten as soon as one later tf_gpu_cache_frame_async() (or any
 * tf_gpu_synchronize / tf_gpu_wait that covers it) has returned -- which is what a lookahead ring
 * needs: a slot is only rewritten by a later av1_lookahead_push (lookahead.c:126,150). */
int tf_gpu_cache_frame_async(tf_gpu_ctx *ctx, const tf_gpu_frame *frame);
/* Same as tf_gpu_cache_frame, but frame->plane[] are DEVICE pointers on the context's device (stride in
 * samples, crop/aligned sizes and frame_id as for host frames; frame->border is ignored: only the crop area is
 * read).  `stream` (a cudaStream_t; NULL = the legacy default stream) is the stream the producer wrote the
 * planes on: the ingest starts after the work already enqueued there, and before returning the call makes
 * `stream` wait for the ingest, so the caller may overwrite or free the planes in stream order.  Never blocks
 * the host.  A frame_id that is already resident with the same geometry is not re-read (same id => same pixels).
 * TF_GPU_ERR_INVALID, with nothing enqueued, for frame_id 0, a NULL plane, bad geometry, a plane that is not
 * device or managed memory of the context's device, or one whose crop area
 * ((crop_h - 1) * stride + crop_w samples from pixel (0,0)) runs past its allocation.  Allocations are those
 * cuMemGetAddressRange reports; where an allocator maps its memory in chunks (virtual-memory mappings, stream-ordered
 * pools), an extent may continue into chunks mapped contiguously after the first one on the same device.  Both
 * chroma planes are read with the one uv stride. */
int tf_gpu_cache_frame_device(tf_gpu_ctx *ctx, const tf_gpu_frame *frame, void *stream);
int tf_gpu_evict_frame(tf_gpu_ctx *ctx, uint64_t frame_id);
/* Test hook for the upload path (av1_copy_and_extend_frame, extend.c:113-163): copies the rectangle
 * [x0, x0+w) x [y0, y0+h) of a cached device plane (coordinates relative to pixel (0,0); negative =
 * border) into dst (samples of the frame's container type, dst_stride in samples).  The rectangle
 * must lie inside the device allocation (tf_gpu_device_border() samples of luma border). */
int tf_gpu_debug_read_plane(tf_gpu_ctx *ctx, uint64_t frame_id, int plane, void *dst, int dst_stride,
                            int x0, int y0, int w, int h);
int tf_gpu_device_border(void);

/* Device-resident variant used by the benchmark's kernel-only number and by the
 * multi-GPU slab mode: frames must already be cached (ids), output stays on the
 * device until tf_gpu_download_output.  time_ms (nullable) receives the CUDA
 * event time of the filter kernel alone. */
int tf_gpu_filter_resident(tf_gpu_ctx *ctx, const tf_gpu_params *params,
                           const uint64_t *frame_ids /*[num_frames]*/,
                           int64_t diff_sum_sse[2], float *time_ms);
/* Asynchronous halves of the above, so that several contexts (independent windows, SURVEY 8e)
 * can be in flight on one GPU: _async enqueues, _result waits and returns FRAME_DIFF / kernel time. */
int tf_gpu_filter_resident_async(tf_gpu_ctx *ctx, const tf_gpu_params *params, const uint64_t *frame_ids);
int tf_gpu_filter_resident_result(tf_gpu_ctx *ctx, int64_t diff_sum_sse[2], float *time_ms);
int tf_gpu_download_output(tf_gpu_ctx *ctx, tf_gpu_frame *out, int row_begin, int row_end);
/* Batched windows: n windows over frames that are already resident, in one call and three kernel launches in all.
 * A frame that several windows read -- the windows centred on every frame of a clip, the KF and ARF windows of one
 * GOP -- is cached once, where one context per window (SURVEY 8e) caches it once per context.  Throughput
 * (DESIGN.md §5): at 640x360 a batch is faster than several contexts in flight (up to +44 % at 16 windows); at
 * 1080p and 4K it is faster than one window after another but 1-17 % slower than several contexts in flight.  Every window has
 * its own params (num_frames, filter_frame_idx, noise levels, q_factor, strength, search settings,
 * compute_frame_diff) and its own device output frame; all frames of a batch share one geometry.
 * frame_ids[w] lists params[w].num_frames ids.  TF_GPU_ERR_INVALID, with nothing enqueued and the context unchanged,
 * for: n outside [1, TF_GPU_MAX_BATCH]; a NULL array; a window that fails the checks of
 * tf_gpu_filter_resident_async (params, ids resident, geometry); frames of different geometry; more distinct
 * frames than the cache holds; a window with out_row_begin / out_row_end or extend_output_borders; an output
 * plane imported with tf_gpu_output_ipc_import; counters enabled (tf_gpu_collect_counters).
 * The batch's outputs are separate from the output of the single-window calls: neither overwrites the other.
 * _result waits for the batch and returns each window's FRAME_DIFF (diff_sum_sse[w], nullable) and the device
 * time of its three kernels.  The outputs stay valid until the next batch of this context. */
#define TF_GPU_MAX_BATCH 16
int tf_gpu_filter_batch_async(tf_gpu_ctx *ctx, int n, const tf_gpu_params *params /*[n]*/,
                              const uint64_t *const *frame_ids /*[n][params[i].num_frames]*/);
int tf_gpu_filter_batch_result(tf_gpu_ctx *ctx, int64_t (*diff_sum_sse)[2] /*[n], nullable*/, float *time_ms);
/* Full blocks of window `window` of the last batch into `out` (as tf_gpu_download_output with all rows); only the
 * window's own params.num_planes planes are written, so a luma-only window needs only out->plane[0]. */
int tf_gpu_download_batch_output(tf_gpu_ctx *ctx, int window, tf_gpu_frame *out);
/* As tf_gpu_output_device_plane, for window `window` of the last batch; TF_GPU_ERR_INVALID for a plane the window
 * does not filter (plane >= its num_planes). */
int tf_gpu_batch_output_device_plane(tf_gpu_ctx *ctx, int window, int plane, void **dptr, size_t *pitch_bytes,
                                     int *rows, int *row_bytes);
/* Raw device pointer + pitch (bytes) of an output plane, for NCCL gathers in
 * slab mode (the reference's counterpart is the shared tf_ctx->output_frame
 * written by all row workers, av1/encoder/ethread.c:2083-2108). */
int tf_gpu_output_device_plane(tf_gpu_ctx *ctx, int plane, void **dptr, size_t *pitch_bytes,
                               int *rows, int *row_bytes);

/* Slab mode over peer memory (one process per GPU on one NVLink / NVSwitch box): the rank that owns the output
 * frame exports its device output planes as CUDA IPC handles; the other ranks import them, and from then on their
 * filter calls store their block rows (out_row_begin/end) straight into the owner's planes over NVLink -- the
 * shared tf_ctx->output_frame all row workers of the reference write (ethread.c:2083-2108), with no gather step.
 * A rank's stores are visible to the owner once its call has completed (tf_gpu_filter_resident_result /
 * tf_gpu_wait) and any inter-process synchronisation (e.g. the FRAME_DIFF all-reduce) has been passed.
 * export: valid after the first filter call of that geometry (the planes exist); handle = 64 opaque bytes
 * (cudaIpcMemHandle_t), offset = byte offset of pixel (0, 0) from the allocation base.
 * import: handle == NULL closes the mapping and returns to the context's own planes; pitch_bytes must equal the
 * importing context's own output pitch for that plane (same frame geometry), checked at the next filter call. */
#define TF_GPU_IPC_HANDLE_BYTES 64
int tf_gpu_output_ipc_export(tf_gpu_ctx *ctx, int plane, unsigned char handle[TF_GPU_IPC_HANDLE_BYTES],
                             size_t *offset_bytes, size_t *pitch_bytes);
int tf_gpu_output_ipc_import(tf_gpu_ctx *ctx, int plane, const unsigned char *handle, size_t offset_bytes,
                             size_t pitch_bytes);

/* First consumer beyond the temporal filter (SURVEY 8f rank 4): the full-pixel search engine as a batch call.
 * Every item is one block of `src` at luma position (x, y) searched in `ref` from a full-pel start MV with
 * av1_full_pixel_search() (mcomp.c:1693-1832; NSTEP sites, cost_list == NULL) configured as tf_motion_search()
 * configures it (temporal_filter.c:145-160: L1 MV cost class from the frame size, mesh search with the
 * prune level / patterns of `params`, skip-row SAD with its audit): the search first_pass_motion_search()
 * (firstpass.c:261-300) and TPL's motion_estimation() (tpl_model.c:285) run per 16x16 / 32x32 block with the
 * same sites.  MV limits are those av1_set_mv_row_limits / av1_set_mv_col_limits (mcomp.h:216-240) give a
 * block of that size at that position, clamped by av1_set_mv_search_range around a zero reference MV.
 * block_size: 16 or 32; x must be a multiple of 16 and y of 4, the block inside the 8-aligned frame.
 * Of `params` the fields bit_depth, mi_rows, mi_cols, cm_width/height, border_in_pixels, prune_mesh_level,
 * mesh_patterns, use_downsampled_sad and q_factor are read.  results[i] = the best full-pel MV and
 * get_mvpred_var_cost() at it, i.e. av1_full_pixel_search()'s return value. */
typedef struct {
  int x, y;                     /* luma position of the block's top-left sample */
  int16_t start_row, start_col; /* full-pel start MV */
} tf_gpu_search_item;
typedef struct {
  int16_t row, col; /* best full-pel MV */
  int32_t var;      /* variance + MV cost at it (INT_MAX when the search was impossible) */
} tf_gpu_search_result;
int tf_gpu_fullpel_search_batch(tf_gpu_ctx *ctx, const tf_gpu_params *params, const tf_gpu_frame *src,
                                const tf_gpu_frame *ref, int block_size, const tf_gpu_search_item *items, int n,
                                tf_gpu_search_result *results);
/* The whole per-block motion search over resident frames, against up to TF_GPU_MAX_FRAMES - 1 references in one
 * launch.  Every item gets what tf_motion_search() (temporal_filter.c:145-188) does to one block of frame src_id
 * searched in frame ref_ids[item.ref], with the MV limits of the item's own size and position (the rule of
 * tf_gpu_fullpel_search_batch): av1_full_pixel_search() from the item's start MV, then find_fractional_mv_step
 * (mcomp.c:2844-3133: MV_COST_NONE, forced_stop = EIGHTH_PEL, no cost list, limits from
 * av1_set_subpel_mv_search_range around a zero MV); under force_integer_mv == 1 there is no sub-pel stage:
 * row, col = 8 x the full-pel MV and err = the variance at it (:162-172).  TPL (tpl_model.c:285) and first pass
 * (firstpass.c:261-300) run this search per 16x16 / 32x32 block against each of their reference frames.
 * Of `params` the fields tf_gpu_fullpel_search_batch reads are read, plus force_integer_mv, allow_hp,
 * subpel_method and subpel_iters_per_step.  src_id and every ref_ids[r] must be resident (tf_gpu_cache_frame*,
 * tf_gpu_cache_frame_device) with one geometry; a reference may repeat or equal the source.  The stream waits
 * for each frame's upload or ingest.  TF_GPU_ERR_INVALID, with nothing enqueued and the context unchanged, for
 * a NULL pointer, block_size other than 16 or 32, n < 0, num_refs outside [1, TF_GPU_MAX_FRAMES - 1], an id
 * that is not resident, frames of different geometry, an item whose position fails the rule above or whose
 * ref is outside [0, num_refs) (the whole call is rejected; tf_gpu_motion_search_device below rejects such an
 * item alone).  n == 0 returns TF_GPU_OK.  Synchronous; tf_gpu_last_stats reports one launch and the search
 * kernel's device time. */
typedef struct {
  int x, y;                     /* luma position of the block's top-left sample */
  int16_t start_row, start_col; /* full-pel start MV */
  int32_t ref;                  /* index into ref_ids */
} tf_gpu_motion_item;
typedef struct {
  int16_t fullpel_row, fullpel_col; /* av1_full_pixel_search() best MV */
  int32_t fullpel_var;              /* its return value (variance + MV cost), as tf_gpu_search_result.var */
  int16_t row, col;                 /* final MV, 1/8 pel */
  uint32_t err;                     /* sub-pel besterr; under force_integer_mv the variance at the full-pel MV */
} tf_gpu_motion_result;
int tf_gpu_motion_search_batch(tf_gpu_ctx *ctx, const tf_gpu_params *params, uint64_t src_id,
                               const uint64_t *ref_ids, int num_refs, int block_size,
                               const tf_gpu_motion_item *items, int n, tf_gpu_motion_result *results);
/* The same search with items and results in DEVICE (or managed) memory of the context's device, ordered on the
 * caller's `stream` (a cudaStream_t; NULL = the legacy default stream): for a caller whose blocks and start MVs are
 * already on the GPU (a torch pipeline; a two-stage search whose 32x32 MVs start the 16x16 blocks), with no round
 * trip through the host between stages.  Params, ids, block size, the fields read and the results are those of
 * tf_gpu_motion_search_batch, bit for bit.  The search starts after the work already enqueued on `stream`, and
 * before returning the call makes `stream` wait for it, so the caller may produce the items and consume or free
 * both buffers in its own stream order.  The search runs on the context's stream, so it also queues behind a filter
 * call already submitted on this context.  Never blocks the host (no synchronise, no host copy, no allocation).
 * TF_GPU_ERR_INVALID, with nothing enqueued and the context unchanged, for what tf_gpu_motion_search_batch rejects
 * before reading its items (NULL pointers, block_size, n < 0, num_refs, residency, geometry), for items or results
 * that are not device or managed memory of the context's device, not 4-byte aligned, or whose n * 16 bytes run past
 * their allocation (checked as tf_gpu_cache_frame_device checks a plane), and for items and results that overlap.
 * n == 0 returns TF_GPU_OK with nothing enqueued.  The host cannot read the items, so the kernel checks each one
 * against the position rule and 0 <= ref < num_refs; where tf_gpu_motion_search_batch rejects the whole call, here
 * only the item is rejected: its result is fullpel_var = TF_GPU_MOTION_REJECTED, MVs 0 and err = UINT32_MAX, and the
 * other items are searched as usual.  tf_gpu_last_stats reports one launch and a kernel time of 0: the call does not
 * wait for the kernel, so it does not time it. */
#define TF_GPU_MOTION_REJECTED (-1) /* fullpel_var of a rejected item; a searched item's is never negative */
int tf_gpu_motion_search_device(tf_gpu_ctx *ctx, const tf_gpu_params *params, uint64_t src_id,
                                const uint64_t *ref_ids /* host */, int num_refs, int block_size,
                                const tf_gpu_motion_item *items /* device */, int n,
                                tf_gpu_motion_result *results /* device */, void *stream);

/* Pinned host memory helpers so lookahead buffers can be DMA'd directly. */
int tf_gpu_host_register(tf_gpu_ctx *ctx, void *ptr, size_t bytes);
int tf_gpu_host_unregister(tf_gpu_ctx *ctx, void *ptr);

/* Launch statistics of the last filter call: number of kernel launches and the
 * device time (ms) of the block-filter kernel. */
int tf_gpu_last_stats(const tf_gpu_ctx *ctx, int *kernel_launches, float *filter_kernel_ms);

/* Executed-work instrumentation for the INT roofline (SURVEY 8d "executed op count"): when
 * enabled, the search kernels count [0] SAD sample pairs read, [1] sub-pel candidate samples,
 * [2] full-pel variance samples of the next filter call(s).  Off by default (atomics perturb timing). */
int tf_gpu_collect_counters(tf_gpu_ctx *ctx, int enable);
int tf_gpu_read_counters(tf_gpu_ctx *ctx, uint64_t counters[4]);

/* Device time (ms) of the three kernels of the last filter call:
 * [0] tf_search32_kernel, [1] tf_search16_kernel, [2] tf_filter_kernel. */
int tf_gpu_last_kernel_times(tf_gpu_ctx *ctx, float ms[3]);

/* Measurement hooks (bench.py): CUDA events recorded on the context's own
 * stream (the stream every kernel of this library is launched on), slots 0..3. */
int tf_gpu_event_record(tf_gpu_ctx *ctx, int slot);
int tf_gpu_event_elapsed_ms(tf_gpu_ctx *ctx, int slot_begin, int slot_end, float *ms);
int tf_gpu_synchronize(tf_gpu_ctx *ctx);
/* Integer-pipe microbenchmark used for the INT roofline denominator
 * (SURVEY 8d): kind 0 = IADD3 (alu pipe), 1 = IMAD (fma pipe),
 * 2 = VABSDIFF4.U8.ACC, 3 = VIMNMX.U16x2, 4 = IDP.4A, 5 = DFMA (fp64).
 * Returns giga warp-lane instructions per second over the whole chip. */
int tf_gpu_microbench(tf_gpu_ctx *ctx, int kind, double *giga_lane_ops_per_s);

#ifdef __cplusplus
}
#endif
#endif /* TF_GPU_H_ */
