/*
 * TEST INFRASTRUCTURE -- see tf_oracle.h.  Scalar C restatement of the
 * reference's temporal-filter hot path.  Every function cites the reference
 * file:line (relative to /root/reference) it follows.  All samples are held as
 * uint16_t here regardless of bit depth; the arithmetic is the reference's.
 *
 * Parity status: PINNED against oracle/_ref (the compiled, unmodified
 * reference) by tests/test_oracle_vs_ref.py and tests/golden/.
 */
#include "tf_oracle.h"

#include <limits.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

#define MINI(a, b) ((a) < (b) ? (a) : (b))
#define MAXI(a, b) ((a) > (b) ? (a) : (b))
#define RPOT(v, n) (((v) + ((1 << (n)) >> 1)) >> (n)) /* aom_ports/mem.h:45 */
static int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }
static int align_pow2(int v, int n) { return (v + (1 << n) - 1) & ~((1 << n) - 1); }

/* Event counters (tf_oracle.h): observe only. */
static tfo_stats g_stats;
static tfo_limit_stats g_lstats;
void tfo_reset_stats(void) { memset(&g_stats, 0, sizeof(g_stats)); memset(&g_lstats, 0, sizeof(g_lstats)); }
void tfo_get_stats(tfo_stats *out) { *out = g_stats; }
void tfo_get_limit_stats(tfo_limit_stats *out) { *out = g_lstats; }

typedef struct { int row, col; } mv_t; /* MV / FULLPEL_MV, av1/common/mv.h:37-47 */

/* ------------------------------------------------------------------------- */
/* Frames: YV12 layout subset (aom_scale/generic/yv12config.c:223-258) with   */
/* borders replicated as av1_copy_and_extend_frame does (extend.c:113-163).   */
/* ------------------------------------------------------------------------- */
typedef struct {
  uint16_t *alloc[3];
  uint16_t *buf[3]; /* pixel (0,0) */
  int stride[2];
  int crop_w[2], crop_h[2];
  int aw[2], ah[2]; /* aligned sizes (widths[]/heights[]) */
  int bw[2], bh[2]; /* border per plane class */
  int rows[2];
} frame_t;

struct tfo_ctx {
  tfo_params p;
  int num_planes, num_pels, mb_rows, mb_cols, mi_rows, mi_cols;
  int min_cm_size; /* AOMMIN(cm->width, cm->height), temporal_filter.c:99-100 */
  frame_t *frames;
  frame_t out;
};

static void frame_alloc(frame_t *f, const tfo_params *p) {
  memset(f, 0, sizeof(*f));
  /* yv12config.c:229-245: aligned_width=(w+7)&~7, y_stride=align32(aw+2*border),
   * uv dims = aligned >> ss, uv_stride = y_stride >> ss_x, uv border = border >> ss */
  const int aw = align_pow2(p->width, 3), ah = align_pow2(p->height, 3);
  /* The frames' own border is border_in_pixels, but at least 64 (AOM_ENC_ALLINTRA_BORDER, the smallest the encoder
   * configures).  Below 64 the MV limits still keep the luma reads inside border_in_pixels, but a chroma predictor
   * at the limit reads (limit >> ss) + 5 samples out, past a (border >> ss) chroma border; the library's frames
   * have a wide replicated border, so the oracle gives those reads replicated samples too. */
  const int border = MAXI(p->border, 64);
  f->aw[0] = aw; f->ah[0] = ah;
  f->aw[1] = aw >> p->ss_x; f->ah[1] = ah >> p->ss_y;
  f->crop_w[0] = p->width; f->crop_h[0] = p->height;
  f->crop_w[1] = (p->width + p->ss_x) >> p->ss_x;
  f->crop_h[1] = (p->height + p->ss_y) >> p->ss_y;
  f->stride[0] = align_pow2(aw + 2 * border, 5);
  f->stride[1] = f->stride[0] >> p->ss_x;
  f->bw[0] = f->bh[0] = border;
  f->bw[1] = border >> p->ss_x; f->bh[1] = border >> p->ss_y;
  const int np = p->monochrome ? 1 : 3;
  for (int pl = 0; pl < np; pl++) {
    const int c = pl > 0;
    f->rows[c] = f->ah[c] + 2 * f->bh[c];
    f->alloc[pl] = (uint16_t *)calloc((size_t)f->rows[c] * f->stride[c], sizeof(uint16_t));
    f->buf[pl] = f->alloc[pl] + (size_t)f->bh[c] * f->stride[c] + f->bw[c];
  }
}
static void frame_free(frame_t *f) { for (int i = 0; i < 3; i++) free(f->alloc[i]); }

/* extend.c:20-65 (copy_and_extend_plane) with the extents of :113-131 (dst->border: the frame's own border) */
static void plane_fill(frame_t *f, int pl, const void *src, int use_hbd, const tfo_params *p) {
  const int c = pl > 0;
  const int w = f->crop_w[c], h = f->crop_h[c], st = f->stride[c];
  const int border = f->bw[0];
  const int er_y = MAXI(f->aw[0] + border, align_pow2(f->aw[0], 6)) - f->crop_w[0];
  const int eb_y = MAXI(f->ah[0] + border, align_pow2(f->ah[0], 6)) - f->crop_h[0];
  const int et = c ? border >> p->ss_y : border;
  const int el = c ? border >> p->ss_x : border;
  const int er = c ? er_y >> p->ss_x : er_y;
  const int eb = c ? eb_y >> p->ss_y : eb_y;
  uint16_t *dst = f->buf[pl];
  for (int y = 0; y < h; y++) {
    uint16_t *row = dst + (size_t)y * st;
    for (int x = 0; x < w; x++)
      row[x] = use_hbd ? ((const uint16_t *)src)[(size_t)y * w + x] : ((const uint8_t *)src)[(size_t)y * w + x];
    for (int x = 1; x <= el; x++) row[-x] = row[0];
    for (int x = 0; x < er; x++) row[w + x] = row[w - 1];
  }
  const int linesize = el + er + w;
  for (int y = 1; y <= et; y++) memcpy(dst - (size_t)y * st - el, dst - el, linesize * 2);
  for (int y = 0; y < eb; y++)
    memcpy(dst + (size_t)(h + y) * st - el, dst + (size_t)(h - 1) * st - el, linesize * 2);
}

tfo_ctx *tfo_create(const tfo_params *p) {
  tfo_ctx *c = (tfo_ctx *)calloc(1, sizeof(*c));
  c->p = *p;
  c->num_planes = p->monochrome ? 1 : 3;
  c->num_pels = 1024 + (p->monochrome ? 0 : 2 * (1024 >> (p->ss_x + p->ss_y)));
  c->mb_rows = (p->height + 31) / 32; /* temporal_filter.c:1236-1237 */
  c->mb_cols = (p->width + 31) / 32;
  tfo_set_coded(c, 0, 0, 0, 0);
  c->frames = (frame_t *)calloc(p->num_frames, sizeof(frame_t));
  for (int i = 0; i < p->num_frames; i++) frame_alloc(&c->frames[i], p);
  frame_alloc(&c->out, p);
  return c;
}
void tfo_set_coded(tfo_ctx *c, int mi_rows, int mi_cols, int cm_width, int cm_height) {
  const tfo_params *p = &c->p;
  /* cm->mi_params (alloccommon.c enc_set_mb_mi: 4-px units of the 8-aligned coded size) unless given */
  c->mi_rows = mi_rows > 0 ? mi_rows : align_pow2(p->height, 3) >> 2;
  c->mi_cols = mi_cols > 0 ? mi_cols : align_pow2(p->width, 3) >> 2;
  /* cm->width / cm->height: the coded size, equal to the crop size unless given */
  const int cm_w = cm_width > 0 ? cm_width : p->width, cm_h = cm_height > 0 ? cm_height : p->height;
  c->min_cm_size = MINI(cm_w, cm_h);
}
void tfo_destroy(tfo_ctx *c) {
  if (!c) return;
  for (int i = 0; i < c->p.num_frames; i++) frame_free(&c->frames[i]);
  frame_free(&c->out);
  free(c->frames);
  free(c);
}
void tfo_set_frame(tfo_ctx *c, int idx, const void *y, const void *u, const void *v) {
  const void *pl[3] = { y, u, v };
  for (int i = 0; i < c->num_planes; i++) plane_fill(&c->frames[idx], i, pl[i], c->p.use_hbd, &c->p);
}
int tfo_get_plane_with_border(tfo_ctx *c, int idx, int plane, uint16_t *dst, int *rows, int *bw, int *bh) {
  frame_t *f = idx < 0 ? &c->out : &c->frames[idx];
  const int k = plane > 0;
  *rows = f->rows[k]; *bw = f->bw[k]; *bh = f->bh[k];
  if (dst) memcpy(dst, f->alloc[plane], (size_t)f->rows[k] * f->stride[k] * 2);
  return f->stride[k];
}
/* aom_extend_frame_borders_c -> extend_frame(ybf, ybf->border) (yv12extend.c): every plane replicated from
 * its crop area, top/left by the border, bottom/right by the border plus aligned - crop */
void tfo_extend_output_borders(tfo_ctx *c) {
  frame_t *f = &c->out;
  for (int pl = 0; pl < c->num_planes; pl++) {
    const int k = pl > 0;
    const int w = f->crop_w[k], h = f->crop_h[k], st = f->stride[k];
    const int et = f->bh[k], el = f->bw[k];
    const int eb = et + f->ah[k] - h, er = el + f->aw[k] - w;
    uint16_t *dst = f->buf[pl];
    for (int y = 0; y < h; y++) {
      uint16_t *row = dst + (size_t)y * st;
      for (int x = 1; x <= el; x++) row[-x] = row[0];
      for (int x = 0; x < er; x++) row[w + x] = row[w - 1];
    }
    const int linesize = el + er + w;
    for (int y = 1; y <= et; y++) memcpy(dst - (size_t)y * st - el, dst - el, linesize * 2);
    for (int y = 0; y < eb; y++)
      memcpy(dst + (size_t)(h + y) * st - el, dst + (size_t)(h - 1) * st - el, linesize * 2);
  }
}
int tfo_plane_alloc_size(tfo_ctx *c, int plane) {
  const int k = plane > 0;
  return c->frames[0].rows[k] * c->frames[0].stride[k];
}
void tfo_get_output(tfo_ctx *c, int plane, uint16_t *dst, int w, int h) {
  const int k = plane > 0;
  for (int y = 0; y < h; y++)
    memcpy(dst + (size_t)y * w, c->out.buf[plane] + (size_t)y * c->out.stride[k], w * 2);
}

/* ------------------------------------------------------------------------- */
/* Noise estimate: temporal_filter.c:1150-1194                                */
/* ------------------------------------------------------------------------- */
static double estimate_noise(const uint16_t *src, int stride, int width, int height, int bd, int edge_thresh) {
  int64_t accum = 0;
  int count = 0;
  for (int i = 1; i < height - 1; ++i) {
    for (int j = 1; j < width - 1; ++j) {
      const uint16_t *m = src + (size_t)i * stride + j;
      const int a = m[-stride - 1], b = m[-stride], c = m[-stride + 1];
      const int d = m[-1], e = m[0], f = m[1];
      const int g = m[stride - 1], h = m[stride], k = m[stride + 1];
      const int Gx = (a - c) + (g - k) + 2 * (d - f);
      const int Gy = (a - g) + (c - k) + 2 * (b - h);
      const int Ga = RPOT(abs(Gx) + abs(Gy), bd - 8);
      if (Ga < edge_thresh) {
        const int v = 4 * e - 2 * (b + h + d + f) + (a + c + g + k);
        accum += RPOT(abs(v), bd - 8);
        ++count;
      }
    }
  }
  return (count < 16) ? -1.0 : (double)accum / (6 * count) * 1.25331413732;
}
/* edge_thresh: NOISE_ESTIMATION_EDGE_THRESHOLD (50, temporal_filter.h:79) unless the caller passes another */
double tfo_estimate_noise_thresh(tfo_ctx *c, int idx, int plane, int edge_thresh) {
  const frame_t *f = &c->frames[idx];
  const int k = plane > 0;
  return estimate_noise(f->buf[plane], f->stride[k], f->crop_w[k], f->crop_h[k], c->p.bit_depth, edge_thresh);
}
double tfo_estimate_noise(tfo_ctx *c, int idx, int plane) { return tfo_estimate_noise_thresh(c, idx, plane, 50); }

/* ------------------------------------------------------------------------- */
/* SAD / variance primitives                                                  */
/* ------------------------------------------------------------------------- */
/* aom_dsp/sad.c:22-36,45-70 (8-bit), :240-304 + encoder_utils.h:152-166,424-436
 * (high bitdepth: >>2 at 10 bit, >>4 at 12 bit after the sum; skip = 2*SAD of
 * even rows, shift applied after the doubling). */
unsigned tfo_sad(const uint16_t *a, int as, const uint16_t *b, int bs, int w, int h, int skip,
                 int bd, int use_hbd) {
  unsigned s = 0;
  const int step = skip ? 2 : 1;
  const int maxd = (1 << (use_hbd ? bd : 8)) - 1;
  for (int y = 0; y < h; y += step) {
    int peak = 0;
    for (int x = 0; x < w; x++) {
      const int d = abs((int)a[y * as + x] - (int)b[y * bs + x]);
      s += d;
      peak += d == maxd;
      if ((x & 15) == 15) { g_stats.sad_peak_groups += peak == 16; peak = 0; }
    }
  }
  if (skip) s *= 2;
  if (use_hbd) s >>= (bd == 10 ? 2 : (bd == 12 ? 4 : 0));
  return s;
}

/* aom_dsp/variance.c:56-72,141-148 (8-bit); :342-429 (high bitdepth).
 * Operand order matters at 10/12 bit because sum is rounded before squaring. */
unsigned tfo_variance(const uint16_t *a, int as, const uint16_t *b, int bs, int w, int h,
                      int bd, int use_hbd, unsigned *sse_out) {
  int64_t sum = 0;
  uint64_t sse = 0;
  for (int y = 0; y < h; y++)
    for (int x = 0; x < w; x++) {
      const int d = (int)a[y * as + x] - (int)b[y * bs + x];
      sum += d;
      sse += (uint32_t)(d * d);
    }
  if (!use_hbd || bd == 8) {
    const uint32_t sse32 = (uint32_t)sse;
    const int s = (int)sum;
    *sse_out = sse32;
    return sse32 - (uint32_t)(((int64_t)s * s) / (w * h));
  }
  const int sh = bd == 10 ? 2 : 4;
  const uint32_t sse32 = (uint32_t)((sse + ((1ull << (2 * sh)) >> 1)) >> (2 * sh));
  const int s = (int)((sum + ((1 << sh) >> 1)) >> sh);
  *sse_out = sse32;
  const int64_t var = (int64_t)sse32 - (((int64_t)s * s) / (w * h));
  return var >= 0 ? (uint32_t)var : 0;
}

/* aom_dsp/variance.c:91-139,150-163 (+ :478-560 hbd), taps aom_filter.h:47-50 */
unsigned tfo_subpel_variance(const uint16_t *ref, int rs, int xoff, int yoff, const uint16_t *src,
                             int ss, int w, int h, int bd, int use_hbd, unsigned *sse) {
  uint16_t fdata3[33 * 32];
  uint16_t temp2[32 * 32];
  const int f0 = 128 - 16 * xoff, f1 = 16 * xoff;
  for (int i = 0; i < h + 1; i++)
    for (int j = 0; j < w; j++)
      fdata3[i * w + j] = (uint16_t)RPOT((int)ref[i * rs + j] * f0 + (int)ref[i * rs + j + 1] * f1, 7);
  const int g0 = 128 - 16 * yoff, g1 = 16 * yoff;
  for (int i = 0; i < h; i++)
    for (int j = 0; j < w; j++) {
      const int v = RPOT((int)fdata3[i * w + j] * g0 + (int)fdata3[(i + 1) * w + j] * g1, 7);
      temp2[i * w + j] = use_hbd ? (uint16_t)v : (uint8_t)v;
    }
  return tfo_variance(temp2, w, src, ss, w, h, bd, use_hbd, sse);
}

/* ------------------------------------------------------------------------- */
/* 12-tap predictor convolve: av1/common/convolve.c:76-174 (8-bit),           */
/* :569-668 (hbd), params convolve.h:63-100, taps filter.h:159-177            */
/* ------------------------------------------------------------------------- */
static const int16_t k12[16][12] = {
  { 0, 0, 0, 0, 0, 128, 0, 0, 0, 0, 0, 0 },
  { 0, 1, -2, 3, -7, 127, 8, -4, 2, -1, 1, 0 },
  { -1, 2, -3, 6, -13, 124, 18, -8, 4, -2, 2, -1 },
  { -1, 3, -4, 8, -18, 120, 28, -12, 7, -4, 2, -1 },
  { -1, 3, -6, 10, -21, 115, 38, -15, 8, -5, 3, -1 },
  { -2, 4, -6, 12, -24, 108, 49, -18, 10, -6, 3, -2 },
  { -2, 4, -7, 13, -25, 100, 60, -21, 11, -7, 4, -2 },
  { -2, 4, -7, 13, -26, 91, 71, -24, 13, -7, 4, -2 },
  { -2, 4, -7, 13, -25, 81, 81, -25, 13, -7, 4, -2 },
  { -2, 4, -7, 13, -24, 71, 91, -26, 13, -7, 4, -2 },
  { -2, 4, -7, 11, -21, 60, 100, -25, 13, -7, 4, -2 },
  { -2, 3, -6, 10, -18, 49, 108, -24, 12, -6, 4, -2 },
  { -1, 3, -5, 8, -15, 38, 115, -21, 10, -6, 3, -1 },
  { -1, 2, -4, 7, -12, 28, 120, -18, 8, -4, 3, -1 },
  { -1, 2, -2, 4, -8, 18, 124, -13, 6, -3, 2, -1 },
  { 0, 1, -1, 2, -4, 8, 127, -7, 3, -2, 1, 0 }
};

static uint16_t clip_px(int v, int bd) { const int m = (1 << bd) - 1; return (uint16_t)(v < 0 ? 0 : (v > m ? m : v)); }
/* clip_px of the predictor, counted */
static uint16_t clip_pred(int v, int bd) {
  g_stats.pred_clip_lo += v < 0;
  g_stats.pred_clip_hi += v > (1 << bd) - 1;
  return clip_px(v, bd);
}

void tfo_convolve12(const uint16_t *src, int ss, uint16_t *dst, int ds, int w, int h,
                    int subpel_x, int subpel_y, int bd, int use_hbd) {
  /* get_conv_params_no_round, convolve.h:63-95: round_0 = 3, round_1 = 11;
   * bd 12: intbufrange = bd+7-3+2 = 18 > 16 -> round_0 = 5, round_1 = 9 */
  int r0 = 3, r1 = 11;
  const int pbd = use_hbd ? bd : 8;
  if (use_hbd && bd + 7 - r0 + 2 > 16) { const int d = bd + 7 - r0 + 2 - 16; r0 += d; r1 -= d; }
  const int fo = 5; /* taps/2 - 1 */
  if (!subpel_x && !subpel_y) { /* aom_convolve_copy */
    for (int y = 0; y < h; y++) memcpy(dst + y * ds, src + y * ss, w * 2);
  } else if (subpel_x && !subpel_y) { /* convolve.c:149-174 / :569-594 */
    const int16_t *f = k12[subpel_x];
    const int bits = 7 - r0;
    for (int y = 0; y < h; y++)
      for (int x = 0; x < w; x++) {
        int32_t res = 0;
        for (int k = 0; k < 12; k++) res += f[k] * src[y * ss + x - fo + k];
        res = RPOT(res, r0);
        dst[y * ds + x] = clip_pred(RPOT(res, bits), pbd);
      }
  } else if (!subpel_x && subpel_y) { /* convolve.c:128-147 / :596-614 */
    const int16_t *f = k12[subpel_y];
    for (int y = 0; y < h; y++)
      for (int x = 0; x < w; x++) {
        int32_t res = 0;
        for (int k = 0; k < 12; k++) res += f[k] * src[(y - fo + k) * ss + x];
        dst[y * ds + x] = clip_pred(RPOT(res, 7), pbd);
      }
  } else { /* convolve.c:76-126 / :616-668 */
    int16_t im[(32 + 11) * 32];
    const int im_h = h + 11;
    const int bits = 14 - r0 - r1;
    const int16_t *fx = k12[subpel_x], *fy = k12[subpel_y];
    const uint16_t *sh = src - fo * ss;
    for (int y = 0; y < im_h; y++)
      for (int x = 0; x < w; x++) {
        int32_t sum = 1 << (pbd + 7 - 1);
        for (int k = 0; k < 12; k++) sum += fx[k] * sh[y * ss + x - fo + k];
        g_stats.conv_im_overflow += RPOT(sum, r0) < INT16_MIN || RPOT(sum, r0) > INT16_MAX;
        im[y * w + x] = (int16_t)RPOT(sum, r0);
      }
    const int ob = pbd + 14 - r0;
    for (int y = 0; y < h; y++)
      for (int x = 0; x < w; x++) {
        int32_t sum = 1 << ob;
        for (int k = 0; k < 12; k++) sum += fy[k] * im[(y + k) * w + x];
        int32_t res = RPOT(sum, r1) - ((1 << (ob - r1)) + (1 << (ob - r1 - 1)));
        if (!use_hbd) res = (int16_t)res; /* convolve.c:120 keeps it in an int16_t */
        dst[y * ds + x] = clip_pred(RPOT(res, bits), pbd);
      }
  }
}

/* tf_build_predictor temporal_filter.c:328-390 with init_subpel_params
 * reconinter.h:131-165 and enc_calc_subpel_params reconinter_enc.c:31-41 */
static void build_predictor(const tfo_ctx *c, const frame_t *ref, int mb_row, int mb_col,
                            const mv_t *mvs, uint16_t *pred) {
  const tfo_params *p = &c->p;
  int plane_offset = 0;
  for (int plane = 0; plane < c->num_planes; plane++) {
    const int ssy = plane ? p->ss_y : 0, ssx = plane ? p->ss_x : 0;
    const int k = plane > 0;
    const int plane_h = 32 >> ssy, plane_w = 32 >> ssx;
    const int plane_y = (32 * mb_row) >> ssy, plane_x = (32 * mb_col) >> ssx;
    const int h = plane_h >> 1, w = plane_w >> 1;
    int idx = 0;
    for (int i = 0; i < plane_h; i += h) {
      for (int j = 0; j < plane_w; j += w) {
        const mv_t mv = mvs[idx++];
        const int y = plane_y + i, x = plane_x + j;
        int pos_y = ((y << 4) + mv.row * (1 << (1 - ssy))) * 64 + 32;
        int pos_x = ((x << 4) + mv.col * (1 << (1 - ssx))) * 64 + 32;
        /* top/left = -(((288 >> ss) - 4) << 10); bottom/right = (dim + 4) << 10,
         * dim = ref_frame->heights/widths (aligned), temporal_filter.c:361-364 */
        const int top = -(((288 >> ssy) - 4) << 10), left = -(((288 >> ssx) - 4) << 10);
        pos_y = clampi(pos_y, top, (ref->ah[k] + 4) << 10);
        pos_x = clampi(pos_x, left, (ref->aw[k] + 4) << 10);
        const uint16_t *src = ref->buf[plane] + (pos_y >> 10) * ref->stride[k] + (pos_x >> 10);
        tfo_convolve12(src, ref->stride[k], &pred[plane_offset + i * plane_w + j], plane_w, w, h,
                       (pos_x & 1023) >> 6, (pos_y & 1023) >> 6, p->bit_depth, p->use_hbd);
      }
    }
    plane_offset += plane_h * plane_w;
  }
}

/* ------------------------------------------------------------------------- */
/* Weights: av1_apply_temporal_filter_c temporal_filter.c:557-707             */
/* ------------------------------------------------------------------------- */
static void apply_filter(int frame_w, int frame_h, int ss_x, int ss_y, int num_planes, int bd,
                         const uint16_t *const src[3], const int stride[2], int mb_row, int mb_col,
                         const double *noise_levels, const mv_t *mvs, const int *mses, int q_factor,
                         int strength, const uint16_t *pred, uint32_t *accum, uint16_t *count) {
  const int min_frame_size = MINI(frame_h, frame_w);
  const double inv_factor = 1.0 / ((5 + 1) * 20);
  const double weight_factor = (double)5 * inv_factor;
  double decay_factor[3] = { 0 };
  double q_decay = pow((double)q_factor / 20, 2);
  q_decay = q_decay < 1e-5 ? 1e-5 : (q_decay > 1 ? 1 : q_decay);
  if (q_factor >= 128) q_decay = 0.5 * pow((double)q_factor / 64, 2);
  double s_decay = pow((double)strength / 4, 2);
  s_decay = s_decay < 1e-5 ? 1e-5 : (s_decay > 1 ? 1 : s_decay);
  for (int plane = 0; plane < num_planes; plane++) {
    const double n_decay = 0.5 + log(2 * noise_levels[plane] + 5.0);
    decay_factor[plane] = 1 / (n_decay * q_decay * s_decay);
  }
  double d_factor[4] = { 0 };
  for (int i = 0; i < 4; i++) {
    const double distance = sqrt(pow(mvs[i].row, 2) + pow(mvs[i].col, 2));
    double thr = min_frame_size * 0.1;
    thr = thr > 1 ? thr : 1;
    d_factor[i] = distance / thr;
    d_factor[i] = d_factor[i] > 1 ? d_factor[i] : 1;
  }
  uint32_t square_diff[1024];
  uint32_t luma_sse_sum[1024];
  memset(square_diff, 0, sizeof(square_diff));
  memset(luma_sse_sum, 0, sizeof(luma_sse_sum));
  int plane_offset = 0;
  for (int plane = 0; plane < num_planes; plane++) {
    const int ssy = plane ? ss_y : 0, ssx = plane ? ss_x : 0;
    const int h = 32 >> ssy, w = 32 >> ssx;
    const int st = stride[plane > 0];
    const int frame_offset = mb_row * h * st + mb_col * w;
    const int num_ref_pixels = 25 + (plane ? (1 << (ssx + ssy)) : 0);
    const double inv_num_ref_pixels = 1.0 / num_ref_pixels;
    if (plane == 1) { /* compute_luma_sq_error_sum :507-522 */
      for (int i = 0; i < h; i++)
        for (int j = 0; j < w; j++)
          for (int ii = 0; ii < (1 << ssy); ii++)
            for (int jj = 0; jj < (1 << ssx); jj++) {
              const int yy = (i << ssy) + ii, xx = (j << ssx) + jj, ww = w << ssx;
              luma_sse_sum[i * w + j] += square_diff[yy * ww + xx];
            }
    }
    for (int i = 0; i < h; i++) /* compute_square_diff :463-493 */
      for (int j = 0; j < w; j++) {
        const int d = (int)src[plane][frame_offset + i * st + j] - (int)pred[plane_offset + i * w + j];
        square_diff[i * w + j] = (uint32_t)(d * d);
      }
    int pred_idx = 0;
    for (int i = 0; i < h; i++) {
      for (int j = 0; j < w; j++) {
        uint64_t sum_square_diff = 0;
        for (int wi = -2; wi <= 2; wi++)
          for (int wj = -2; wj <= 2; wj++) {
            const int y = clampi(i + wi, 0, h - 1), x = clampi(j + wj, 0, w - 1);
            sum_square_diff += square_diff[y * w + x];
          }
        sum_square_diff += luma_sse_sum[i * w + j];
        if (bd > 8) sum_square_diff >>= ((bd - 8) * 2);
        const double window_error = sum_square_diff * inv_num_ref_pixels;
        const int sb = (i >= h / 2) * 2 + (j >= w / 2);
        const double block_error = (double)mses[sb];
        const double combined_error = weight_factor * window_error + block_error * inv_factor;
        double scaled_error = combined_error * d_factor[sb] * decay_factor[plane];
        scaled_error = scaled_error < 7 ? scaled_error : 7;
        const int weight = (int)(exp(-scaled_error) * 1000);
        const int idx = plane_offset + pred_idx;
        accum[idx] += weight * pred[idx];
        count[idx] += weight;
        ++pred_idx;
      }
    }
    plane_offset += h * w;
  }
}

void tfo_apply_block(int width, int height, int ss_x, int ss_y, int num_planes, int bd, int use_hbd,
                     const void *src_y, const void *src_u, const void *src_v, int y_stride,
                     int uv_stride, int mb_row, int mb_col, const double *noise_levels,
                     const int16_t *mvs, const int *mses, int q_factor, int strength,
                     const void *pred, uint32_t *accum, uint16_t *count) {
  /* widen everything to u16 */
  const void *sp[3] = { src_y, src_u, src_v };
  uint16_t *planes[3] = { 0, 0, 0 };
  int stride[2] = { y_stride, uv_stride };
  for (int pl = 0; pl < num_planes; pl++) {
    const int ssy = pl ? ss_y : 0, ssx = pl ? ss_x : 0;
    const int h = 32 >> ssy, w = 32 >> ssx, st = stride[pl > 0];
    const size_t n = (size_t)(mb_row * h + h) * st + mb_col * w + w;
    planes[pl] = (uint16_t *)malloc(n * 2);
    for (size_t i = 0; i < n; i++)
      planes[pl][i] = use_hbd ? ((const uint16_t *)sp[pl])[i] : ((const uint8_t *)sp[pl])[i];
  }
  int num_pels = 1024 + (num_planes > 1 ? 2 * (1024 >> (ss_x + ss_y)) : 0);
  uint16_t *p16 = (uint16_t *)malloc(num_pels * 2);
  for (int i = 0; i < num_pels; i++)
    p16[i] = use_hbd ? ((const uint16_t *)pred)[i] : ((const uint8_t *)pred)[i];
  mv_t m[4];
  for (int i = 0; i < 4; i++) { m[i].row = mvs[2 * i]; m[i].col = mvs[2 * i + 1]; }
  const uint16_t *cs[3] = { planes[0], planes[1], planes[2] };
  apply_filter(width, height, ss_x, ss_y, num_planes, bd, cs, stride, mb_row, mb_col, noise_levels,
               m, mses, q_factor, strength, p16, accum, count);
  for (int pl = 0; pl < 3; pl++) free(planes[pl]);
  free(p16);
}

/* aom_dsp/odintrin.h:30-42: table multiply-shift for d < 1024, else x / d.
 * tests/test_oracle_vs_ref.py proves OD_DIVU(x,d) == x/d exhaustively for
 * d in [1000,1023], x <= 21000*4095+10500 against the compiled reference. */
int tfo_od_divu(unsigned x, unsigned d) { return (int)(x / d); }

/* ------------------------------------------------------------------------- */
/* Motion search                                                              */
/* ------------------------------------------------------------------------- */
typedef struct { int col_min, col_max, row_min, row_max; } limits_t;

typedef struct {
  /* NSTEP site table, mcomp.c:433-475 */
  mv_t site[15][13];
  int searches_per_step[15];
  int radius[15];
} sites_t;

static void init_nstep(sites_t *s) {
  int radius = 1;
  for (int st = 0; st < 15; st++) {
    int tan_radius = MAXI((int)(0.41 * radius), 1);
    int n = 12;
    if (radius <= 5) { tan_radius = radius; n = 8; }
    const mv_t m[13] = {
      { 0, 0 }, { -radius, 0 }, { radius, 0 }, { 0, -radius }, { 0, radius },
      { -radius, -tan_radius }, { radius, tan_radius }, { -tan_radius, radius },
      { tan_radius, -radius }, { -radius, tan_radius }, { radius, -tan_radius },
      { tan_radius, radius }, { -tan_radius, -radius },
    };
    for (int i = 0; i <= n; i++) s->site[st][i] = m[i];
    s->searches_per_step[st] = n;
    s->radius[st] = radius;
    if (st < 12) radius = (int)MAXI((radius * 1.5 + 0.5), radius + 1);
  }
}

typedef struct {
  const tfo_params *p;
  const uint16_t *src; /* block in the frame to filter */
  const uint16_t *ref; /* co-located block in the reference frame */
  int stride;
  int w, h;       /* 32x32 or 16x16 */
  int use_skip;   /* sdf == sdsf */
  limits_t lim;   /* full-pel */
  int sad_lambda, sse_lambda; /* mcomp.c:237-244 */
  const sites_t *sites;
  int min_frame_size;
} search_t;

/* GET_MV_RAWPEL, mv.h:28 */
static int rawpel(int x) { return (x + 3 + (x >= 0)) >> 3; }

static unsigned s_sad(const search_t *s, int r, int c, int skip) {
  return tfo_sad(s->src, s->stride, s->ref + r * s->stride + c, s->stride, s->w, s->h, skip,
                 s->p->bit_depth, s->p->use_hbd);
}
/* mvsad_err_cost mcomp.c:310-331, ref = 0, L1 */
static int sad_cost(const search_t *s, int r, int c) { return (s->sad_lambda * (abs(r * 8) + abs(c * 8))) >> 3; }
/* mv_err_cost mcomp.c:271-295 on a 1/8-pel mv, ref = 0 */
static int sse_cost(const search_t *s, int r8, int c8) { return (s->sse_lambda * (abs(r8) + abs(c8))) >> 3; }
/* get_mvpred_var_cost / get_mvpred_compound_var_cost mcomp.c:645-708: vf(src, ref) */
static int var_cost(const search_t *s, int r, int c) {
  unsigned sse;
  int v = (int)tfo_variance(s->src, s->stride, s->ref + r * s->stride + c, s->stride, s->w, s->h,
                            s->p->bit_depth, s->p->use_hbd, &sse);
  return v + sse_cost(s, r * 8, c * 8);
}
static int in_range(const limits_t *l, int r, int c) {
  return c >= l->col_min && c <= l->col_max && r >= l->row_min && r <= l->row_max;
}

/* clamp_fullmv, as diamond_search_sad and exhaustive_mesh_search call it on their start MV: clamp() tests the low
 * bound first (v < lo ? lo : v > hi ? hi : v), so the high bound wins when the limits invert.  Counted. */
static mv_t clamp_start(const limits_t *l, mv_t mv) {
  const mv_t c = { clampi(mv.row, l->row_min, l->row_max), clampi(mv.col, l->col_min, l->col_max) };
  g_lstats.start_clamped += c.row != mv.row || c.col != mv.col;
  return c;
}

/* diamond_search_sad mcomp.c:1299-1416 */
static unsigned diamond_search(const search_t *s, mv_t start, int search_step, int skip, int *num00,
                               mv_t *best_mv) {
  const sites_t *cfg = s->sites;
  start = clamp_start(&s->lim, start);
  const int tot_steps = 15 - search_step;
  *num00 = 0;
  *best_mv = start;
  unsigned bestsad = s_sad(s, start.row, start.col, skip) + sad_cost(s, start.row, start.col);
  int is_off_center = 0;
  int next_step_size = tot_steps > 2 ? cfg->radius[tot_steps - 2] : 1;
  for (int step = tot_steps - 1; step >= 0; --step) {
    const mv_t *site = cfg->site[step];
    int best_site = 0;
    if (step > 0) next_step_size = cfg->radius[step - 1];
    int all_in = 1;
    all_in &= best_mv->row + site[1].row >= s->lim.row_min;
    all_in &= best_mv->row + site[2].row <= s->lim.row_max;
    all_in &= best_mv->col + site[3].col >= s->lim.col_min;
    all_in &= best_mv->col + site[4].col <= s->lim.col_max;
    for (int idx = 1; idx <= cfg->searches_per_step[step]; idx++) {
      const int r = best_mv->row + site[idx].row, c = best_mv->col + site[idx].col;
      if (!all_in && !in_range(&s->lim, r, c)) continue;
      unsigned thissad = s_sad(s, r, c, skip);
      g_stats.diamond_ties += thissad + sad_cost(s, r, c) == bestsad;
      if (thissad < bestsad) {
        thissad += sad_cost(s, r, c);
        if (thissad < bestsad) { bestsad = thissad; best_site = idx; }
      }
    }
    if (best_site != 0) {
      best_mv->row += site[best_site].row;
      best_mv->col += site[best_site].col;
      is_off_center = 1;
    }
    if (is_off_center == 0) (*num00)++;
    if (best_site == 0) {
      while (next_step_size == cfg->radius[step] && step > 2) {
        ++(*num00);
        --step;
        next_step_size = cfg->radius[step - 1];
      }
    }
  }
  return bestsad;
}

/* full_pixel_diamond mcomp.c:1421-1470 (cost_list == NULL) */
static int full_pixel_diamond(const search_t *s, mv_t start, int step_param, int skip, mv_t *best_mv) {
  int n, num00 = 0;
  int bestsme = (int)diamond_search(s, start, step_param, skip, &n, best_mv);
  if (bestsme < INT_MAX) bestsme = var_cost(s, best_mv->row, best_mv->col);
  const int further_steps = 15 - 1 - step_param;
  while (n < further_steps) {
    ++n;
    if (num00) {
      num00--;
    } else {
      mv_t tmp;
      int thissme = (int)diamond_search(s, start, step_param + n, skip, &num00, &tmp);
      if (thissme < INT_MAX) thissme = var_cost(s, tmp.row, tmp.col);
      if (thissme < bestsme) { bestsme = thissme; *best_mv = tmp; }
    }
  }
  return bestsme;
}

/* update_mvs_and_sad mcomp.c:839-858 */
static void upd(const search_t *s, unsigned this_sad, int r, int c, unsigned *best_sad, mv_t *best) {
  g_stats.mesh_ties += this_sad + sad_cost(s, r, c) == *best_sad;
  if (this_sad >= *best_sad) return;
  const unsigned sad = this_sad + sad_cost(s, r, c);
  if (sad < *best_sad) { *best_sad = sad; best->row = r; best->col = c; }
}

/* exhaustive_mesh_search mcomp.c:1474-1543 */
static int mesh_search(const search_t *s, mv_t start, int range, int step, int skip, mv_t *best_mv) {
  const int col_step = (step > 1) ? step : 4;
  start = clamp_start(&s->lim, start);
  *best_mv = start;
  unsigned best_sad = s_sad(s, start.row, start.col, skip) + sad_cost(s, start.row, start.col);
  const int start_row = MAXI(-range, s->lim.row_min - start.row);
  const int start_col = MAXI(-range, s->lim.col_min - start.col);
  const int end_row = MINI(range, s->lim.row_max - start.row);
  const int end_col = MINI(range, s->lim.col_max - start.col);
  for (int r = start_row; r <= end_row; r += step) {
    for (int c = start_col; c <= end_col; c += col_step) {
      if (step > 1) {
        upd(s, s_sad(s, start.row + r, start.col + c, skip), start.row + r, start.col + c, &best_sad, best_mv);
      } else if (c + 3 <= end_col) {
        for (int i = 0; i < 4; ++i)
          upd(s, s_sad(s, start.row + r, start.col + c + i, skip), start.row + r, start.col + c + i, &best_sad, best_mv);
      } else {
        for (int i = 0; i < end_col - c; ++i) /* sic: end_col itself is never visited */
          upd(s, s_sad(s, start.row + r, start.col + c + i, skip), start.row + r, start.col + c + i, &best_sad, best_mv);
      }
    }
  }
  return (int)best_sad;
}

/* full_pixel_exhaustive mcomp.c:1547-1617 */
static int full_pixel_exhaustive(const search_t *s, mv_t start, int skip, mv_t *best_mv) {
  const tfo_params *p = s->p;
  int interval = p->mesh[0][1], range = p->mesh[0][0];
  *best_mv = start;
  if (range < 7 || range > 256 || interval < 1 || interval > range) return INT_MAX;
  g_stats.mesh_searches++;
  const int baseline_interval_divisor = range / interval;
  range = MAXI(range, (5 * MAXI(abs(best_mv->row), abs(best_mv->col))) / 4);
  range = MINI(range, 256);
  interval = MAXI(interval, range / baseline_interval_divisor);
  int bestsme = mesh_search(s, *best_mv, range, interval, skip, best_mv);
  if (interval > 1 && range > 7) {
    for (int i = 1; i < 4; ++i) {
      bestsme = mesh_search(s, *best_mv, p->mesh[i][0], p->mesh[i][1], skip, best_mv);
      if (p->mesh[i][1] == 1) break;
    }
  }
  if (bestsme < INT_MAX) bestsme = var_cost(s, best_mv->row, best_mv->col);
  return bestsme;
}

/* av1_full_pixel_search mcomp.c:1693-1832, NSTEP, run_mesh_search = 1 */
static int full_pixel_search(const search_t *s, mv_t start, int step_param, int skip, mv_t *best_mv) {
  const tfo_params *p = s->p;
  int run_mesh = 1;
  int var = full_pixel_diamond(s, start, step_param, skip, best_mv);
  /* prune: mcomp.c:138-140 (LVL_2, thr 4), temporal_filter.c:152-156 (LVL_1: q>20, thr 2) */
  int prune = 0, thr = 4;
  if (p->prune_mesh_level == 2) prune = 1;
  if (p->prune_mesh_level == 1) { prune = (p->q_factor <= 20) ? 0 : 1; thr = 2; }
  if (prune) {
    const int d = MAXI(abs(start.row - best_mv->row), abs(start.col - best_mv->col));
    if (d <= thr) run_mesh = 0;
  }
  if (skip) { /* mcomp.c:1777-1810 */
    const int sad = (int)s_sad(s, best_mv->row, best_mv->col, 0);
    const int skip_sad = (int)s_sad(s, best_mv->row, best_mv->col, 1);
    const int kSADThresh = s->w * s->h / 16; /* 1 << (mi_w_log2 + mi_h_log2) */
    if (sad > kSADThresh && abs(skip_sad - sad) * 10 >= MAXI(sad, 1) * 9)
      return full_pixel_search(s, start, step_param, 0, best_mv);
  }
  if (run_mesh) {
    mv_t tmp;
    const int var_ex = full_pixel_exhaustive(s, *best_mv, skip, &tmp);
    if (var_ex < var) { var = var_ex; *best_mv = tmp; }
  }
  return var;
}

/* ---- sub-pel ------------------------------------------------------------ */
typedef struct {
  const search_t *s;
  limits_t lim; /* sub-pel limits, mcomp.h:344-361 */
  unsigned besterr;
  mv_t best;
} subpel_t;

/* aom_upsampled_pred_c reconinter_enc.c:424-496 (+ highbd :656-730) with
 * EIGHTTAP_REGULAR (av1_get_filter(USE_8_TAPS), filter.h:270-279), via
 * aom_convolve8_horiz/vert_c aom_dsp/aom_convolve.c:36-72 (8-bit intermediate)
 * and aom_highbd_convolve8_* :118-180.  Then vf(pred, w, src) mcomp.c:2385,2405 */
static const int16_t k8[16][8] = { /* av1_sub_pel_filters_8, filter.h:123-133 */
  { 0, 0, 0, 128, 0, 0, 0, 0 },      { 0, 2, -6, 126, 8, -2, 0, 0 },
  { 0, 2, -10, 122, 18, -4, 0, 0 },  { 0, 2, -12, 116, 28, -8, 2, 0 },
  { 0, 2, -14, 110, 38, -10, 2, 0 }, { 0, 2, -14, 102, 48, -12, 2, 0 },
  { 0, 2, -16, 94, 58, -12, 2, 0 },  { 0, 2, -14, 84, 66, -12, 2, 0 },
  { 0, 2, -14, 76, 76, -14, 2, 0 },  { 0, 2, -12, 66, 84, -14, 2, 0 },
  { 0, 2, -12, 58, 94, -16, 2, 0 },  { 0, 2, -12, 48, 102, -14, 2, 0 },
  { 0, 2, -10, 38, 110, -14, 2, 0 }, { 0, 2, -8, 28, 116, -12, 2, 0 },
  { 0, 0, -4, 18, 122, -10, 2, 0 },  { 0, 0, -2, 8, 126, -6, 2, 0 }
};

static unsigned upsampled_err(const search_t *s, int r8, int c8, unsigned *sse) {
  const int w = s->w, h = s->h, st = s->stride;
  const int bd = s->p->use_hbd ? s->p->bit_depth : 8;
  const uint16_t *ref = s->ref + (r8 >> 3) * st + (c8 >> 3);
  const int sx = c8 & 7, sy = r8 & 7;
  uint16_t pred[32 * 32];
  if (!sx && !sy) {
    for (int i = 0; i < h; i++) memcpy(pred + i * w, ref + i * st, w * 2);
  } else if (!sy) {
    const int16_t *k = k8[sx << 1];
    for (int y = 0; y < h; y++)
      for (int x = 0; x < w; x++) {
        int sum = 0;
        for (int t = 0; t < 8; t++) sum += ref[y * st + x - 3 + t] * k[t];
        pred[y * w + x] = clip_px(RPOT(sum, 7), bd);
      }
  } else if (!sx) {
    const int16_t *k = k8[sy << 1];
    for (int y = 0; y < h; y++)
      for (int x = 0; x < w; x++) {
        int sum = 0;
        for (int t = 0; t < 8; t++) sum += ref[(y - 3 + t) * st + x] * k[t];
        pred[y * w + x] = clip_px(RPOT(sum, 7), bd);
      }
  } else {
    uint16_t temp[(32 + 7) * 32];
    const int ih = h + 7; /* (((h-1)*8 + sy) >> 3) + 8 */
    const int16_t *kx = k8[sx << 1], *ky = k8[sy << 1];
    for (int y = 0; y < ih; y++)
      for (int x = 0; x < w; x++) {
        int sum = 0;
        for (int t = 0; t < 8; t++) sum += ref[(y - 3) * st + x - 3 + t] * kx[t];
        temp[y * w + x] = clip_px(RPOT(sum, 7), bd);
      }
    for (int y = 0; y < h; y++)
      for (int x = 0; x < w; x++) {
        int sum = 0;
        for (int t = 0; t < 8; t++) sum += temp[(y + t) * w + x] * ky[t];
        pred[y * w + x] = clip_px(RPOT(sum, 7), bd);
      }
  }
  return tfo_variance(pred, w, s->src, st, w, h, s->p->bit_depth, s->p->use_hbd, sse);
}

/* estimated_pref_error mcomp.c:2308-2336: svf(ref@floor(mv/8), mv&7, src) */
static unsigned bilinear_err(const search_t *s, int r8, int c8, unsigned *sse) {
  const uint16_t *ref = s->ref + (r8 >> 3) * s->stride + (c8 >> 3);
  return tfo_subpel_variance(ref, s->stride, c8 & 7, r8 & 7, s->src, s->stride, s->w, s->h,
                             s->p->bit_depth, s->p->use_hbd, sse);
}

/* check_better_fast mcomp.c:2433-2461 / check_better :2465-2488 (MV_COST_NONE) */
static unsigned check_better(subpel_t *sp, int r8, int c8, int accurate, int *is_better) {
  if (!in_range(&sp->lim, r8, c8)) return INT_MAX;
  unsigned sse;
  const unsigned cost = accurate ? upsampled_err(sp->s, r8, c8, &sse) : bilinear_err(sp->s, r8, c8, &sse);
  g_stats.subpel_ties += cost == sp->besterr;
  if (cost < sp->besterr) {
    sp->besterr = cost;
    sp->best.row = r8; sp->best.col = c8;
    if (is_better) *is_better |= 1;
  }
  return cost;
}

/* first_level_check(_fast) mcomp.c:2503-2541, 2626-2660; get_best_diag_step :2490-2498 */
static mv_t first_level(subpel_t *sp, mv_t t, int hstep, int accurate) {
  const unsigned left = check_better(sp, t.row, t.col - hstep, accurate, NULL);
  const unsigned right = check_better(sp, t.row, t.col + hstep, accurate, NULL);
  const unsigned up = check_better(sp, t.row - hstep, t.col, accurate, NULL);
  const unsigned down = check_better(sp, t.row + hstep, t.col, accurate, NULL);
  const mv_t diag = { up <= down ? -hstep : hstep, left <= right ? -hstep : hstep };
  check_better(sp, t.row + diag.row, t.col + diag.col, accurate, NULL);
  return diag;
}

/* second_level_check_fast mcomp.c:2545-2605 */
static void second_level_fast(subpel_t *sp, mv_t t, mv_t diag, int hstep) {
  const int tr = t.row, tc = t.col, br = sp->best.row, bc = sp->best.col;
  if (tr != br && tc != bc) {
    check_better(sp, br, bc + diag.col, 0, NULL);
    check_better(sp, br + diag.row, bc, 0, NULL);
  } else if (tr == br && tc != bc) {
    check_better(sp, br + hstep, bc + diag.col, 0, NULL);
    check_better(sp, br - hstep, bc + diag.col, 0, NULL);
    check_better(sp, br - diag.row, bc, 0, NULL);
  } else if (tr != br && tc == bc) {
    check_better(sp, br + diag.row, bc + hstep, 0, NULL);
    check_better(sp, br + diag.row, bc - hstep, 0, NULL);
    check_better(sp, br, bc - diag.col, 0, NULL);
  }
}

/* second_level_check_v2 mcomp.c:2665-2715 (subpel_search_type = USE_8_TAPS) */
static void second_level_v2(subpel_t *sp, mv_t t, mv_t diag) {
  if (t.row == sp->best.row && t.col == sp->best.col) return;
  if (t.row == sp->best.row) diag.row *= -1;
  else if (t.col == sp->best.col) diag.col *= -1;
  const mv_t rb = { sp->best.row + diag.row, sp->best.col };
  const mv_t cb = { sp->best.row, sp->best.col + diag.col };
  const mv_t db = { sp->best.row + diag.row, sp->best.col + diag.col };
  int has_better = 0;
  check_better(sp, rb.row, rb.col, 1, &has_better);
  check_better(sp, cb.row, cb.col, 1, &has_better);
  if (has_better) check_better(sp, db.row, db.col, 1, &has_better);
}

/* av1_find_best_sub_pixel_tree{,_pruned,_pruned_more} mcomp.c:2844-3133 with
 * cost_list == NULL, forced_stop = EIGHTH_PEL, MV_COST_NONE, unscaled.
 * Returns besterr; *best in 1/8 pel. */
static unsigned subpel_search(const search_t *s, mv_t start_full, mv_t *best) {
  const tfo_params *p = s->p;
  subpel_t sp;
  sp.s = s;
  /* av1_set_subpel_mv_search_range mcomp.h:344-361, ref_mv = 0 */
  const int max_mv = 1023 * 8;
  sp.lim.col_min = MAXI(-(1 << 14) + 1, MAXI(s->lim.col_min * 8, -max_mv));
  sp.lim.col_max = MINI((1 << 14) - 1, MINI(s->lim.col_max * 8, max_mv));
  sp.lim.row_min = MAXI(-(1 << 14) + 1, MAXI(s->lim.row_min * 8, -max_mv));
  sp.lim.row_max = MINI((1 << 14) - 1, MINI(s->lim.row_max * 8, max_mv));
  mv_t start = { start_full.row * 8, start_full.col * 8 };
  sp.best = start;
  unsigned sse;
  int hstep = 4;
  if (p->subpel_method == 0) { /* SUBPEL_TREE :3065-3133 */
    sp.besterr = upsampled_err(s, start.row, start.col, &sse);
    const int round = MINI(3, 3 - !p->allow_hp);
    for (int iter = 0; iter < round; ++iter) {
      const mv_t center = sp.best;
      const mv_t diag = first_level(&sp, center, hstep, 1);
      if (!(center.row == sp.best.row && center.col == sp.best.col) && p->subpel_iters_per_step > 1)
        second_level_v2(&sp, center, diag);
      hstep >>= 1;
    }
  } else { /* PRUNED (:2929) and PRUNED_MORE (:2844) coincide when cost_list == NULL */
    /* setup_center_error :2718-2777: vf(ref, src) */
    sp.besterr = tfo_variance(s->ref + start_full.row * s->stride + start_full.col, s->stride, s->src,
                              s->stride, s->w, s->h, p->bit_depth, p->use_hbd, &sse);
    const int rounds = p->allow_hp ? 3 : 2;
    for (int it = 0; it < rounds; it++) {
      const mv_t center = sp.best;
      const mv_t diag = first_level(&sp, center, hstep, 0);
      if (p->subpel_iters_per_step > 1) second_level_fast(&sp, center, diag, hstep);
      hstep >>= 1;
    }
  }
  *best = sp.best;
  return sp.besterr;
}

/* av1_set_mv_{row,col}_limits mcomp.h:216-240 + av1_set_mv_search_range
 * mcomp.c:196-215 with ref_mv = 0 */
static void set_limits(const tfo_ctx *c, int mi_row, int mi_col, int mi_size, limits_t *l) {
  const int border = c->p.border;
  const int mih = mi_size, miw = mi_size;
  /* cm->mi_params: c->mi_rows / c->mi_cols (the coded grid) */
  const int b_row_min = -(mi_row * 4 + border - 8), b_row_max = (c->mi_rows - mi_row - mih) * 4 + border - 8;
  const int b_col_min = -(mi_col * 4 + border - 8), b_col_max = (c->mi_cols - mi_col - miw) * 4 + border - 8;
  const int e_row_min = -(((mi_row + mih) * 4) + 8), e_row_max = (c->mi_rows - mi_row) * 4 + 8;
  const int e_col_min = -(((mi_col + miw) * 4) + 8), e_col_max = (c->mi_cols - mi_col) * 4 + 8;
  l->row_min = MAXI(b_row_min, e_row_min);
  l->row_max = MINI(b_row_max, e_row_max);
  l->col_min = MAXI(b_col_min, e_col_min);
  l->col_max = MINI(b_col_max, e_col_max);
  /* ref_mv = 0: [-1023, 1023] intersect (MV_LOW/8+1.. never binds) */
  l->col_min = MAXI(l->col_min, -1023); l->col_max = MINI(l->col_max, 1023);
  l->row_min = MAXI(l->row_min, -1023); l->row_max = MINI(l->row_max, 1023);
  /* counters only */
  g_lstats.lim_inverted += l->row_min > l->row_max || l->col_min > l->col_max;
  g_lstats.lim_border_bound += (b_row_min > e_row_min && b_row_min > -1023) || (b_row_max < e_row_max && b_row_max < 1023) ||
                              (b_col_min > e_col_min && b_col_min > -1023) || (b_col_max < e_col_max && b_col_max < 1023);
}

/* tf_motion_search temporal_filter.c:94-130: the search state of one frame pair; returns step_param */
static int search_setup(const tfo_ctx *c, const sites_t *sites, int stride, search_t *s, int *skip) {
  const tfo_params *p = &c->p;
  /* :99-100 min_frame_size = AOMMIN(cm->width, cm->height): the coded size */
  const int min_frame_size = c->min_cm_size;
  memset(s, 0, sizeof(*s));
  s->p = p;
  s->stride = stride;
  s->sites = sites;
  s->min_frame_size = min_frame_size;
  /* :119-122 MV_COST_L1_{HDRES,MIDRES,LOWRES} by min_frame_size, mcomp.c:237-244 */
  if (min_frame_size >= 720) { s->sad_lambda = 8; s->sse_lambda = 1; }
  else if (min_frame_size >= 480) { s->sad_lambda = 15; s->sse_lambda = 0; }
  else { s->sad_lambda = 32; s->sse_lambda = 2; }
  /* use_downsampled_sad && block_size_high >= 16: true for both sizes */
  *skip = p->use_downsampled_sad ? 1 : 0;
  /* av1_init_search_range mcomp.c:217-226 of the larger crop dimension of the frame to filter (not cm->width) */
  int size = MAXI(16, MAXI(p->width, p->height));
  int step_param = 0;
  while ((size << step_param) < 1023) step_param++;
  return MINI(step_param, 9);
}

void tfo_full_pixel_search(tfo_ctx *c, int src_idx, int ref_idx, int bsize, int x, int y,
                           int start_row, int start_col, int *out) {
  sites_t sites;
  init_nstep(&sites);
  const frame_t *cur = &c->frames[src_idx], *ref = &c->frames[ref_idx];
  const int st = cur->stride[0];
  search_t s;
  int skip;
  const int step_param = search_setup(c, &sites, st, &s, &skip);
  set_limits(c, y >> 2, x >> 2, bsize >> 2, &s.lim);
  s.src = cur->buf[0] + (size_t)y * st + x;
  s.ref = ref->buf[0] + (size_t)y * st + x;
  s.w = s.h = bsize;
  const mv_t start = { start_row, start_col };
  mv_t best;
  out[2] = full_pixel_search(&s, start, step_param, skip, &best);
  out[0] = best.row;
  out[1] = best.col;
}

/* counters only: a full-pel MV on a search limit, and whether the +-1023 clamp set that limit */
static void count_on_limit(const limits_t *l, mv_t mv) {
  const int rl = mv.row == l->row_min || mv.row == l->row_max;
  const int cl = mv.col == l->col_min || mv.col == l->col_max;
  g_stats.mv_on_limit += rl || cl;
  g_stats.mv_on_clamp += (mv.row == -1023 || mv.row == 1023 || mv.col == -1023 || mv.col == 1023) && (rl || cl);
}

/* tf_motion_search temporal_filter.c:87-253 */
static void motion_search(const tfo_ctx *c, const sites_t *sites, const frame_t *cur, const frame_t *ref,
                          int mb_row, int mb_col, mv_t *ref_mv, mv_t *sub_mvs, int *sub_mses) {
  const tfo_params *p = &c->p;
  const int st = cur->stride[0];
  const int y_offset = mb_row * 32 * st + mb_col * 32;
  const int min_frame_size = c->min_cm_size; /* :99-100, AOMMIN(cm->width, cm->height) */
  search_t s;
  int skip;
  const int step_param = search_setup(c, sites, st, &s, &skip);
  set_limits(c, mb_row * 8, mb_col * 8, 8, &s.lim);

  mv_t start = { rawpel(ref_mv->row), rawpel(ref_mv->col) };
  s.src = cur->buf[0] + y_offset;
  s.ref = ref->buf[0] + y_offset;
  s.w = s.h = 32;
  mv_t best_full;
  full_pixel_search(&s, start, step_param, skip, &best_full);
  count_on_limit(&s.lim, best_full);
  int block_mse;
  mv_t block_mv;
  if (p->force_integer_mv == 1) {
    unsigned sse;
    const unsigned err = tfo_variance(s.ref + best_full.row * st + best_full.col, st, s.src, st, 32, 32,
                                      p->bit_depth, p->use_hbd, &sse);
    block_mse = (int)((err + 512) / 1024);
    block_mv.row = best_full.row * 8; block_mv.col = best_full.col * 8;
  } else {
    mv_t best;
    unsigned err = subpel_search(&s, best_full, &best);
    block_mse = (int)((err + 512) / 1024);
    block_mv = best;
    *ref_mv = best;
    start.row = rawpel(ref_mv->row); start.col = rawpel(ref_mv->col);
    int idx = 0;
    for (int i = 0; i < 32; i += 16)
      for (int j = 0; j < 32; j += 16) {
        s.src = cur->buf[0] + y_offset + i * st + j;
        s.ref = ref->buf[0] + y_offset + i * st + j;
        s.w = s.h = 16;
        full_pixel_search(&s, start, step_param, skip, &best_full);
        count_on_limit(&s.lim, best_full);
        err = subpel_search(&s, best_full, &best);
        sub_mses[idx] = (int)((err + 128) / 256);
        sub_mvs[idx] = best;
        ++idx;
      }
  }
  /* tf_determine_block_partition :270-292 */
  int mn = INT_MAX, mx = INT_MIN;
  int64_t sum = 0;
  for (int i = 0; i < 4; i++) { sum += sub_mses[i]; mn = MINI(mn, sub_mses[i]); mx = MAXI(mx, sub_mses[i]); }
  if ((((int64_t)block_mse * 15 < sum * 4) && mx - mn < 48) ||
      (((int64_t)block_mse * 14 < sum * 4) && mx - mn < 24)) {
    for (int i = 0; i < 4; i++) { sub_mvs[i] = block_mv; sub_mses[i] = block_mse; }
  }
  const int thresh = (min_frame_size >= 720) ? 12 : 3; /* :249-250 */
  g_stats.block_mse_at_thresh += block_mse == (thresh << (p->bit_depth - 8));
  if (block_mse > (thresh << (p->bit_depth - 8))) { ref_mv->row = 0; ref_mv->col = 0; g_stats.ref_mv_resets++; }
}

/* av1_tf_do_filtering_row temporal_filter.c:788-939 for rows [row_begin,row_end) */
void tfo_run(tfo_ctx *c, int row_begin, int row_end, int16_t *mvs_out, int32_t *mses_out,
             uint16_t *pred_out, uint32_t *accum_out, uint16_t *count_out, int64_t *diff) {
  const tfo_params *p = &c->p;
  sites_t sites;
  init_nstep(&sites);
  const frame_t *cur = &c->frames[p->filter_frame_idx];
  const int np = c->num_pels;
  uint32_t *accum = (uint32_t *)malloc(np * 4);
  uint16_t *count = (uint16_t *)malloc(np * 2);
  uint16_t *pred = (uint16_t *)malloc(np * 2);
  int64_t dsum = 0, dsse = 0;
  for (int mb_row = row_begin; mb_row < row_end; mb_row++) {
    for (int mb_col = 0; mb_col < c->mb_cols; mb_col++) {
      const int blk = mb_row * c->mb_cols + mb_col;
      memset(accum, 0, np * 4);
      memset(count, 0, np * 2);
      mv_t ref_mv = { 0, 0 };
      for (int frame = 0; frame < p->num_frames; frame++) {
        mv_t sub_mvs[4] = { { 0, 0 }, { 0, 0 }, { 0, 0 }, { 0, 0 } };
        int sub_mses[4] = { INT_MAX, INT_MAX, INT_MAX, INT_MAX };
        if (frame == p->filter_frame_idx) {
          ref_mv.row *= -1; ref_mv.col *= -1;
          /* tf_apply_temporal_filter_self :406-446 */
          int off = 0;
          for (int pl = 0; pl < c->num_planes; pl++) {
            const int h = 32 >> (pl ? p->ss_y : 0), w = 32 >> (pl ? p->ss_x : 0), st = cur->stride[pl > 0];
            const uint16_t *b = cur->buf[pl] + mb_row * h * st + mb_col * w;
            for (int i = 0; i < h; i++)
              for (int j = 0; j < w; j++) { accum[off + i * w + j] += 1000 * b[i * st + j]; count[off + i * w + j] += 1000; }
            off += h * w;
          }
          continue;
        }
        const frame_t *ref = &c->frames[frame];
        motion_search(c, &sites, cur, ref, mb_row, mb_col, &ref_mv, sub_mvs, sub_mses);
        build_predictor(c, ref, mb_row, mb_col, sub_mvs, pred);
        const size_t bf = (size_t)blk * p->num_frames + frame;
        if (mvs_out) for (int i = 0; i < 4; i++) { mvs_out[(bf * 4 + i) * 2] = (int16_t)sub_mvs[i].row; mvs_out[(bf * 4 + i) * 2 + 1] = (int16_t)sub_mvs[i].col; }
        if (mses_out) for (int i = 0; i < 4; i++) mses_out[bf * 4 + i] = sub_mses[i];
        if (pred_out) memcpy(pred_out + bf * np, pred, np * 2);
        const uint16_t *srcp[3] = { cur->buf[0], cur->buf[1], cur->buf[2] };
        apply_filter(p->width, p->height, p->ss_x, p->ss_y, c->num_planes, p->bit_depth, srcp, cur->stride,
                     mb_row, mb_col, p->noise_levels, sub_mvs, sub_mses, p->q_factor, p->filter_strength,
                     pred, accum, count);
      }
      /* tf_normalize_filtered_frame :740-777 */
      int off = 0;
      for (int pl = 0; pl < c->num_planes; pl++) {
        const int h = 32 >> (pl ? p->ss_y : 0), w = 32 >> (pl ? p->ss_x : 0), st = c->out.stride[pl > 0];
        uint16_t *b = c->out.buf[pl] + mb_row * h * st + mb_col * w;
        for (int i = 0; i < h; i++)
          for (int j = 0; j < w; j++) {
            const int idx = off + i * w + j;
            b[i * st + j] = (uint16_t)tfo_od_divu(accum[idx] + (count[idx] >> 1), count[idx]);
          }
        off += h * w;
      }
      if (accum_out) memcpy(accum_out + (size_t)blk * np, accum, np * 4);
      if (count_out) memcpy(count_out + (size_t)blk * np, count, np * 2);
      if (p->compute_frame_diff) { /* :921-937: vf(src, out) */
        unsigned sse;
        tfo_variance(cur->buf[0] + mb_row * 32 * cur->stride[0] + mb_col * 32, cur->stride[0],
                     c->out.buf[0] + mb_row * 32 * c->out.stride[0] + mb_col * 32, c->out.stride[0], 32, 32,
                     p->bit_depth, p->use_hbd, &sse);
        dsum += sse;
        dsse += sse * (int64_t)sse;
      }
    }
  }
  if (diff) { diff[0] = dsum; diff[1] = dsse; }
  free(accum); free(count); free(pred);
}
