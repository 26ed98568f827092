/*
 * TEST INFRASTRUCTURE -- the temporal filter's predictor of one block at a caller MV, composed from the oracle's pinned
 * tfo_convolve12.  The oracle source is compiled into this unit unchanged, so tfo_convolve12 and the frames here are
 * the very code that tests/test_oracle_vs_ref.py pins to the reference; tfo_predict_block restates the position rule of
 * the oracle's build_predictor for one block.  Built by tests/_oracle_predict.py into a temporary directory; the
 * product never links or loads it.
 */
#include "../oracle/tf_oracle.c"

/* The filter's predictor of one block at caller MV (mv_row, mv_col) in 1/8 pel: what build_predictor makes with four
 * equal sub-block MVs, for a bsize x bsize block (16: one luma sub-block and its chroma sub-blocks; 32: the four
 * quadrants, each from its own origin) at luma (x, y) of frame ref_idx.  Position and clamp are build_predictor's
 * (init_subpel_params, temporal_filter.c:356-365); the samples are read through a clamp of the coordinates to the
 * crop area, which is what the frame's edge-replicated border holds, so that every int16 MV is defined however far
 * it reaches.  dst: num_pels = bsize^2 (+ 2 (bsize >> ss_x)(bsize >> ss_y) for num_planes 3) samples in the layout
 * of tfo_run's pred recorder. */
void tfo_predict_block(tfo_ctx *c, int ref_idx, int bsize, int x, int y, int mv_row, int mv_col, int num_planes,
                       uint16_t *dst) {
  const tfo_params *p = &c->p;
  const frame_t *ref = &c->frames[ref_idx];
  int plane_offset = 0;
  for (int plane = 0; plane < num_planes; plane++) {
    const int ssy = plane ? p->ss_y : 0, ssx = plane ? p->ss_x : 0;
    const int k = plane > 0;
    const int plane_h = bsize >> ssy, plane_w = bsize >> ssx;
    const int h = 16 >> ssy, w = 16 >> ssx;
    for (int i = 0; i < plane_h; i += h) {
      for (int j = 0; j < plane_w; j += w) {
        const int py = (y >> ssy) + i, px = (x >> ssx) + j;
        int pos_y = ((py << 4) + mv_row * (1 << (1 - ssy))) * 64 + 32;
        int pos_x = ((px << 4) + mv_col * (1 << (1 - ssx))) * 64 + 32;
        const int top = -(((288 >> ssy) - 4) << 10), left = -(((288 >> ssx) - 4) << 10);
        pos_y = clampi(pos_y, top, (ref->ah[k] + 4) << 10);
        pos_x = clampi(pos_x, left, (ref->aw[k] + 4) << 10);
        const int oy = pos_y >> 10, ox = pos_x >> 10;
        /* the 12-tap footprint [o - 5, o + extent + 6) of each axis, read through the crop clamp */
        uint16_t patch[(16 + 11) * (16 + 11)];
        const int pw = w + 11;
        for (int r = 0; r < h + 11; r++)
          for (int q = 0; q < pw; q++)
            patch[r * pw + q] = ref->buf[plane][(size_t)clampi(oy - 5 + r, 0, ref->crop_h[k] - 1) * ref->stride[k] +
                                                clampi(ox - 5 + q, 0, ref->crop_w[k] - 1)];
        tfo_convolve12(patch + 5 * pw + 5, pw, &dst[plane_offset + i * plane_w + j], plane_w, w, h,
                       (pos_x & 1023) >> 6, (pos_y & 1023) >> 6, p->bit_depth, p->use_hbd);
      }
    }
    plane_offset += plane_h * plane_w;
  }
}
