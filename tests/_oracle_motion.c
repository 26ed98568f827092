/*
 * TEST INFRASTRUCTURE -- the per-block motion search of tf_motion_search() (temporal_filter.c:145-188) composed
 * from the oracle's pinned search routines.  The oracle source is compiled into this unit unchanged, so the
 * static full_pixel_search / subpel_search / set_limits / search_setup used here are the very code that
 * tests/test_oracle_vs_ref.py pins to the reference; nothing of tfo_run changes.  Built by tests/_oracle_motion.py
 * into a temporary directory; the product never links or loads it.
 */
#include "../oracle/tf_oracle.c"

/* tfo_full_pixel_search, then find_fractional_mv_step (MV_COST_NONE, forced_stop = EIGHTH_PEL, no cost list, limits
 * from av1_set_subpel_mv_search_range around a zero MV) from its result, or under force_integer_mv the variance
 * at the full-pel MV (:162-172).  out = full row, full col, full var cost, row (1/8 pel), col (1/8 pel), err. */
void tfo_motion_search(tfo_ctx *c, int src_idx, int ref_idx, int bsize, int x, int y, int start_row,
                       int start_col, int *out) {
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
  mv_t best_full, best;
  out[2] = full_pixel_search(&s, start, step_param, skip, &best_full);
  out[0] = best_full.row;
  out[1] = best_full.col;
  unsigned err;
  if (c->p.force_integer_mv == 1) {
    unsigned sse;
    err = tfo_variance(s.ref + best_full.row * st + best_full.col, st, s.src, st, bsize, bsize, c->p.bit_depth,
                       c->p.use_hbd, &sse);
    best.row = best_full.row * 8;
    best.col = best_full.col * 8;
  } else {
    err = subpel_search(&s, best_full, &best);
  }
  out[3] = best.row;
  out[4] = best.col;
  out[5] = (int)err;
}
