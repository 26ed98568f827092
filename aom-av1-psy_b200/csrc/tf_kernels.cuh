// Device code of the B200 temporal filter.  Hand-written CUDA for sm_100a.
//
// The per-block loop of av1_tf_do_filtering_row (temporal_filter.c:788-939) is
// cut along its real data dependencies into three kernels, each small enough
// for the 32 KB instruction cache (the single fused kernel of the first version
// stalled 54% of its issue slots on instruction fetch):
//   tf_search32_kernel  32x32 search of every frame, chained through ref_mv
//                       (:855-871): one warp per block;
//   tf_search16_kernel  the 16x16 sub-block searches: one warp per independent
//                       (frame, block, sub-block) task -- 56x more parallelism
//                       than blocks for a 15-frame window;
//   tf_filter_kernel    partition decision, 12-tap predictor, weights,
//                       accumulate/count, normalise, FRAME_DIFF: four warps per
//                       block; pred / accum / count never leave shared memory.
// Every data-dependent decision of the reference's search is replayed
// warp-uniformly (all lanes take the same branch after a shuffle reduction), so
// motion vectors are bit-exact by construction.
//
// Integer work is byte/halfword SIMD-in-word: VABSDIFF4.U8.ACC (__vsadu4) for
// 8-bit SAD, VIMNMX.U16x2 (max-min) for high-bitdepth SAD, one IMAD per two
// samples for the bilinear taps, IDP.2A for sums / sums of squares.  No tensor
// cores: nothing on this path is a dense contraction.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace tfk {

constexpr unsigned FULL = 0xffffffffu;
// TF_PU16: near passes of the 16x16 search whose loads are issued back to back (2: 63.5 -> 63.9 frames/s at 4K 10-bit).
#ifndef TF_PU16
#define TF_PU16 2
#endif
// Inlining policy: every search routine is inlined into its kernel.  A routine that is not inlined re-materialises
// the global-memory descriptor for each of its loads (LDC + 2 x R2UR per LDG: 10% of the executed instructions of
// both search kernels in the round-1 build) and passes its context through the stack; the out-of-line routines
// were a round-1 answer to the instruction-fetch stalls of one fused kernel, and with three kernels inlining
// lowers them instead (16x16 search: no_inst 12% -> 5%).  Only the 8-tap routine of SUBPEL_TREE stays out of line.
constexpr int MAXF = 24;
constexpr int INT_MAX_ = 0x7fffffff;

// NSTEP site table (mcomp.c:433-475), built on the host.
struct Sites {
  int16_t r[15][13];
  int16_t c[15][13];
  int32_t n[15];
  int32_t radius[15];
};
__constant__ Sites c_sites;
// MULTITAP_SHARP2 12-tap kernels (av1/common/filter.h:159-177) and
// EIGHTTAP_REGULAR (filter.h:123-133) -- numeric tables of the AV1 format.
__constant__ int16_t c_k12[16][12];
__constant__ int16_t c_k8[16][8];

struct KParams {
  // geometry
  int width, height;  // luma crop
  int mb_rows, mb_cols, mi_rows, mi_cols;
  int ss_x, ss_y, num_planes, bit_depth, is_hbd;
  int aligned_w[2], aligned_h[2];
  int border;  // oxcf.border_in_pixels
  int num_frames, filter_idx;
  int q_factor, strength;
  int force_integer_mv, allow_hp, subpel_method, iters_per_step;
  int prune_level, mesh[4][2], use_skip, compute_diff;
  int sad_lambda, sse_lambda, step_param, mse_thresh;
  int hbd_shift;  // 0, 2 (10 bit), 4 (12 bit): SAD >>, variance rounding
  int row_begin, row_end;
  double decay[3];
  double dist_thr;  // max(min(w,h) * 0.1, 1)
  // planes (pointers to pixel (0,0)); pitch in samples
  const void *frm[MAXF][3];
  const uint16_t *rs[MAXF];  // per frame: luma row sums at pixel (0,0), luma pitch (rowsum16_kernel); 16x16 search
  int pitch[2];
  void *out[3];
  int out_pitch[2];
  unsigned long long *diff;  // [2]
  unsigned long long *ctr;   // [4] optional executed-work counters, see Search::ctr
  // optional dumps (device)
  int16_t *d_mvs;
  int32_t *d_mses;
  uint16_t *d_pred;
  uint32_t *d_accum;  // optional dump of the final accumulators [blocks][num_pels]
  uint16_t *d_count;
  // search results, [blocks][num_frames] and [blocks][num_frames][4] (device scratch)
  int16_t *s_ref_mv;   // [blocks][2]: the ref_mv chain state between per-frame search32 launches
  int frame_begin, frame_end;  // frames [begin, end) handled by this search launch
  int16_t *s_blk_mv;   // 32x32 result (row, col) in 1/8 pel
  int32_t *s_blk_mse;
  int16_t *s_sub_mv;   // 16x16 results
  int32_t *s_sub_mse;
  int num_pels;
};

struct MV2 {
  int row, col;
};
struct Lim {
  int col_min, col_max, row_min, row_max;
};

__device__ __forceinline__ int lane_id() {
  // %laneid through non-volatile asm: the compiler may reuse one read per function instead of issuing an S2R
  // at every inlined use (3% of the executed instructions of the 16x16 search)
  int l;
  asm("mov.u32 %0, %%laneid;" : "=r"(l));
  return l;
}
__device__ __forceinline__ int iabs(int x) { return x < 0 ? -x : x; }
__device__ __forceinline__ int imin(int a, int b) { return a < b ? a : b; }
__device__ __forceinline__ int imax(int a, int b) { return a > b ? a : b; }
__device__ __forceinline__ int iclamp(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }
__device__ __forceinline__ int rpot(int v, int n) { return (v + ((1 << n) >> 1)) >> n; }

template <int N>
__device__ __forceinline__ unsigned seg_reduce_u32(unsigned v) {
#pragma unroll
  for (int o = N / 2; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
  return v;
}
__device__ __forceinline__ unsigned long long warp_sum_u64(unsigned long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
  return v;
}

// Warp sum of a per-lane (sum, sse) pair with one 64-bit reduction: |sum| <= 32 * 4095 < 2^17 per
// lane, so sum + 2^17 is non-negative and the 32-lane total stays below 2^23; sse totals < 2^35.
__device__ __forceinline__ unsigned long long warp_sum_pair(int &sum, unsigned sse) {
  unsigned long long v = ((unsigned long long)sse << 24) | (unsigned)(sum + (1 << 17));
  v = warp_sum_u64(v);
  sum = (int)(v & 0xffffffu) - (1 << 22);
  return v >> 24;
}

// ---------------------------------------------------------------------------
// Search context (warp-uniform)
// ---------------------------------------------------------------------------
template <typename T>
struct Search {
  const T *src;  // block origin in the frame to filter
  const T *ref;  // co-located origin in the reference frame
  int stride;    // samples
  Lim lim;       // full-pel limits
  int sad_lambda, sse_lambda;
  int hbd_shift;
  int is_hbd;
  // Shared-memory search window: the reference samples needed by every
  // candidate whose full-pel MV lies within +-wR of (wr, wc).  Candidates inside
  // are read from shared memory (one conflict-free wavefront per load), the rest
  // from global memory through L1.
  unsigned char *win;  // nullptr = no window
  unsigned srcs;       // shared address of the source-block tile (SrcTile layout), 0 = not staged
  int wr, wc, wR;
  int wpitch;  // bytes; wpitch/4 is odd
  int wshift;  // bytes the window origin was aligned down by
  // optional executed-work counters (bench instrumentation; nullptr in normal runs):
  // [0] SAD sample pairs read, [1] sub-pel candidate evaluations x block samples, [2] variance samples,
  // [3] diamond sites skipped by the row-sum bound
  unsigned long long *ctr;
  // Row sums of the reference (16x16 search only): rs[i * stride + j] = sum of ref[i * stride + j + t], t < 16.
  // nullptr = no row-sum bound.
  const uint16_t *rs;
};

constexpr int WIN_BYTES = 9472;  // window capacity per warp, 32x32 search
constexpr int WIN16_BYTES = 4608;  // 16x16 search (R = 12): lets >= 24 warps share an SM

// SAD lane layout: a candidate occupies LPC lanes (one block row per lane, every
// other row with skip-row SAD, aom_dsp/sad.c:66-70), so a pass evaluates
// CPP = 32 / LPC candidates at once.
template <typename T, int W, bool SKIP>
struct SadL {
  static constexpr int ROWS = SKIP ? W / 2 : W;
  static constexpr int LPC = ROWS;
  static constexpr int CPP = 32 / LPC;
  static constexpr int NW = W * (int)sizeof(T) / 4;
  static constexpr int RSTEP = SKIP ? 2 : 1;
  static constexpr int MAXP = 12 / CPP;  // passes for a 12-site stage
};

// Largest window radius that fits WIN_BYTES for a W x W block of T.
template <typename T, int W>
struct WinCfg {
  static constexpr int R = (W == 32) ? 16 : 12;
  static constexpr int ROWS = W + 2 * R;
  static constexpr int ROWB = ((W + 2 * R) * (int)sizeof(T) + 15 + 15) / 16 * 16;  // + align-down slack, 16B chunks
  static constexpr int PITCH = ROWB + 4 + ((((ROWB + 4) / 4) & 1) ? 0 : 4);         // words per row odd
  static_assert(ROWS * PITCH <= (W == 32 ? WIN_BYTES : WIN16_BYTES), "search window does not fit");
};

// The block of the frame to filter as a shared-memory tile for the sub-pel stage: W rows, row pitch chosen so
// that the row bands of the error routines below fall into disjoint banks.
template <typename T, int W>
struct SrcTile {
  static constexpr int PITCH = sizeof(T) == 2 ? (W == 32 ? 68 : 40) : (W == 32 ? 36 : 20);  // bytes
  static constexpr int BYTES = W * PITCH;
};
// Dynamic shared memory of a search kernel: the window, then the source tile.
template <typename T, int W>
struct SearchSmem {
  static constexpr int WIN = (WinCfg<T, W>::ROWS * WinCfg<T, W>::PITCH + 15) / 16 * 16;
  static constexpr int TOTAL = WIN + SrcTile<T, W>::BYTES;
  static_assert((W + 7) * W * (int)sizeof(T) <= WIN, "8-tap scratch of SUBPEL_TREE lives in the window buffer");
};
template <typename T, int W>
__device__ __forceinline__ void src_tile_load(Search<T> &S, unsigned char *buf) {
  constexpr int ES = (int)sizeof(T), CPR = W * ES / 16, TOTAL = W * CPR;  // 16-byte chunks
  const int lane = lane_id();
  const unsigned char *g = reinterpret_cast<const unsigned char *>(S.src);
  const size_t gpitch = (size_t)S.stride * ES;
#pragma unroll
  for (int q0 = 0; q0 < TOTAL; q0 += 32) {
    const int q = q0 + lane, row = q / CPR, ch = q - row * CPR;
    if (q < TOTAL) {
      const uint4 v = __ldg(reinterpret_cast<const uint4 *>(g + row * gpitch) + ch);
      uint32_t *d = reinterpret_cast<uint32_t *>(buf + row * SrcTile<T, W>::PITCH + ch * 16);
      d[0] = v.x;
      d[1] = v.y;
      d[2] = v.z;
      d[3] = v.w;
    }
  }
  __syncwarp();
  S.srcs = (unsigned)__cvta_generic_to_shared(buf);
}

// Cooperative, coalesced window fill: 16-byte global loads, 4-byte shared stores.
template <typename T, int W>
__device__ __forceinline__ void window_load(Search<T> &S, unsigned char *buf, int wr, int wc) {
  using C = WinCfg<T, W>;
  const int lane = lane_id();
  const T *g0 = S.ref + (wr - C::R) * S.stride + (wc - C::R);
  const uintptr_t a = reinterpret_cast<uintptr_t>(g0);
  const int shift = (int)(a & 15);
  const unsigned char *ga = reinterpret_cast<const unsigned char *>(a - shift);
  constexpr int CPR = C::ROWB / 16;  // chunks per row
  const size_t gpitch = (size_t)S.stride * sizeof(T);
  __syncwarp();
  constexpr int TOTAL = C::ROWS * CPR;
#pragma unroll 1
  for (int q0 = 0; q0 < TOTAL; q0 += 32 * 4) {
    uint4 v[4];
#pragma unroll
    for (int u = 0; u < 4; u++) {  // four independent 16-byte loads in flight per lane
      const int q = q0 + u * 32 + lane;
      const int row = q / CPR, ch = q - row * CPR;
      if (q < TOTAL) v[u] = __ldg(reinterpret_cast<const uint4 *>(ga + row * gpitch + ch * 16));
    }
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const int q = q0 + u * 32 + lane;
      const int row = q / CPR, ch = q - row * CPR;
      if (q < TOTAL) {
        uint32_t *d = reinterpret_cast<uint32_t *>(buf + row * C::PITCH + ch * 16);
        d[0] = v[u].x;
        d[1] = v[u].y;
        d[2] = v[u].z;
        d[3] = v[u].w;
      }
    }
  }
  __syncwarp();
  S.win = buf;
  S.wr = wr;
  S.wc = wc;
  S.wR = C::R;
  S.wpitch = C::PITCH;
  S.wshift = shift;
}

template <typename T, int W, bool SKIP>
__device__ __forceinline__ void sad_load_src(const T *src, int stride, uint32_t (&sw)[SadL<T, W, SKIP>::NW]) {
  using L = SadL<T, W, SKIP>;
  const int row = (lane_id() % L::LPC) * L::RSTEP;
  const uint4 *p = reinterpret_cast<const uint4 *>(src + row * stride);
#pragma unroll
  for (int j = 0; j < L::NW / 4; j++) {
    const uint4 v = __ldg(p + j);
    sw[4 * j + 0] = v.x;
    sw[4 * j + 1] = v.y;
    sw[4 * j + 2] = v.z;
    sw[4 * j + 3] = v.w;
  }
}

// Where the candidates of one diamond stage / mesh level are read from: the
// shared-memory window or global memory.  Uniform per stage, so there is a single
// code path (generic loads) and no per-candidate test.
struct SadSrc {
  const unsigned char *base;  // address of the sample at full-pel MV (0, 0), row 0
  int pitchB;                 // bytes per row
};
template <typename T>
__device__ __forceinline__ SadSrc sad_src(const Search<T> &S, bool use_window) {
  SadSrc q;
  if (use_window) {
    q.base = S.win + ((S.wR - S.wr) * S.wpitch + (S.wR - S.wc) * (int)sizeof(T) + S.wshift);
    q.pitchB = S.wpitch;
  } else {
    q.base = reinterpret_cast<const unsigned char *>(S.ref);
    q.pitchB = S.stride * (int)sizeof(T);
  }
  return q;
}
// All MVs within +-reach of (r, c) lie inside the window.
template <typename T>
__device__ __forceinline__ bool window_covers(const Search<T> &S, int r, int c, int reach) {
  return S.win != nullptr && iabs(r - S.wr) + reach <= S.wR && iabs(c - S.wc) + reach <= S.wR;
}

// Partial SAD of this lane's row (row = lane's block row) of the candidate at full-pel (r, c).
template <typename T, int W, bool SKIP>
__device__ __forceinline__ unsigned sad_partial(const SadSrc &Q, const unsigned char *safe, int r, int c, int row,
                                                bool valid, const uint32_t (&sw)[SadL<T, W, SKIP>::NW]) {
  using L = SadL<T, W, SKIP>;
  const unsigned char *pb = valid ? Q.base + (r + row) * Q.pitchB + c * (int)sizeof(T) : safe;
  const uintptr_t a = reinterpret_cast<uintptr_t>(pb);
  const uint32_t *wp = reinterpret_cast<const uint32_t *>(a & ~(uintptr_t)3);
  const unsigned sh = (unsigned)(a & 3) * 8;
  uint32_t w[L::NW + 1];
#pragma unroll
  for (int j = 0; j <= L::NW; j++) w[j] = wp[j];
  unsigned s = 0;
  if (sizeof(T) == 1) {
#pragma unroll
    for (int j = 0; j < L::NW; j++) s = __vsadu4(__funnelshift_r(w[j], w[j + 1], sh), sw[j]) + s;
  } else {
    unsigned acc = 0;  // two u16 lanes; NW <= 16 words of <= 4095 each: no carry
#pragma unroll
    for (int j = 0; j < L::NW; j++) {
      const unsigned x = __funnelshift_r(w[j], w[j + 1], sh);
      acc += __vmaxu2(x, sw[j]) - __vminu2(x, sw[j]);
    }
    s = (acc & 0xffffu) + (acc >> 16);
  }
  return s;
}

// Same, for candidates inside the shared-memory window: 32-bit shared addresses and
// ld.shared (no generic-address descriptor traffic), branch-free.
__device__ __forceinline__ uint32_t lds_u32(unsigned addr) {
  uint32_t v;
  asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ uint32_t lds_u16(unsigned addr) {
  uint32_t v;
  asm("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}
template <typename T, int W, bool SKIP>
__device__ __forceinline__ unsigned sad_partial_win(unsigned win_origin /* shared addr of MV (0,0), row 0 */,
                                                    int wpitch, int r, int c, int row,
                                                    const uint32_t (&sw)[SadL<T, W, SKIP>::NW], unsigned sa = 0) {
  using L = SadL<T, W, SKIP>;
  const unsigned a = win_origin + (unsigned)((r + row) * wpitch + c * (int)sizeof(T));
  const unsigned wa = a & ~3u, sh = (a & 3u) * 8;
  uint32_t w[L::NW + 1];
#pragma unroll
  for (int j = 0; j <= L::NW; j++) w[j] = lds_u32(wa + 4 * j);
  unsigned s = 0;
  if (sizeof(T) == 1) {
#pragma unroll
    for (int j = 0; j < L::NW; j++) s = __vsadu4(__funnelshift_r(w[j], w[j + 1], sh), sw[j]) + s;
  } else {
    // |a - b| = a + b - 2 min(a, b): the sum of the source row (sa) is known, the candidate's sum and the sum of
    // the minima come from IDP.2A on the FMA pipe -- one VIMNMX on the ALU pipe per word instead of two plus the add
    // (the ALU pipe is the busier one: 54% in the 16x16 search, the FMA pipe 16%; 4K 10-bit 62.5 -> 63.4 frames/s)
    unsigned accb = 0, accm = 0;
#pragma unroll
    for (int j = 0; j < L::NW; j++) {
      const unsigned x = __funnelshift_r(w[j], w[j + 1], sh);
      accb = __dp2a_lo(x, 0x0101u, accb);
      accm = __dp2a_lo(__vminu2(x, sw[j]), 0x0101u, accm);
    }
    s = sa + accb - 2 * accm;
  }
  return s;
}

// mvsad_err_cost (mcomp.c:310-331), L1, ref = 0
template <typename T>
__device__ __forceinline__ int sad_cost(const Search<T> &S, int r, int c) {
  return S.sad_lambda * (iabs(r) + iabs(c));  // == (lambda * (|8r| + |8c|)) >> 3 exactly
}
// mv_err_cost (mcomp.c:271-295) on a 1/8-pel mv
template <typename T>
__device__ __forceinline__ int sse_cost(const Search<T> &S, int r8, int c8) {
  return (S.sse_lambda * (iabs(r8) + iabs(c8))) >> 3;
}
__device__ __forceinline__ bool in_range(const Lim &l, int r, int c) {
  return (c >= l.col_min) & (c <= l.col_max) & (r >= l.row_min) & (r <= l.row_max);  // branch-free
}
template <bool SKIP>
__device__ __forceinline__ unsigned sad_post(unsigned s, int hbd_shift) {
  if (SKIP) s *= 2;
  return s >> hbd_shift;
}

// SAD of one candidate, result in all lanes.
template <typename T, int W, bool SKIP>
__device__ __forceinline__ unsigned sad_single(const Search<T> &S, int r, int c, int lane,
                                               const uint32_t (&sw)[SadL<T, W, SKIP>::NW]) {
  using L = SadL<T, W, SKIP>;
  const SadSrc Q = sad_src(S, window_covers(S, r, c, 0));
  unsigned part = sad_partial<T, W, SKIP>(Q, reinterpret_cast<const unsigned char *>(S.src), r, c,
                                          (lane % L::LPC) * L::RSTEP, true, sw);
  part = seg_reduce_u32<L::LPC>(part);
  return sad_post<SKIP>(part, S.hbd_shift);
}

// Sums four per-lane values over the warp with 6 shuffles instead of 20: after
// two exchange steps every lane owns one of the four values (index
// ((lane >> 4) & 1) * 2 + ((lane >> 3) & 1)), three butterfly steps finish it.
__device__ __forceinline__ unsigned reduce4_u32(const unsigned (&a)[4], int lane) {
  const bool hi16 = lane & 16, hi8 = lane & 8;
  unsigned x0 = hi16 ? a[2] : a[0], y0 = hi16 ? a[0] : a[2];
  unsigned x1 = hi16 ? a[3] : a[1], y1 = hi16 ? a[1] : a[3];
  x0 += __shfl_xor_sync(FULL, y0, 16);
  x1 += __shfl_xor_sync(FULL, y1, 16);
  unsigned x = hi8 ? x1 : x0, y = hi8 ? x0 : x1;
  x += __shfl_xor_sync(FULL, y, 8);
  x += __shfl_xor_sync(FULL, x, 4);
  x += __shfl_xor_sync(FULL, x, 2);
  x += __shfl_xor_sync(FULL, x, 1);
  return x;
}

template <int FROM>
__device__ __forceinline__ unsigned group_min_u32(unsigned v) {  // min across lane groups of FROM lanes
#pragma unroll
  for (int o = FROM; o < 32; o <<= 1) v = min(v, __shfl_xor_sync(FULL, v, o));
  return v;
}

// ---------------------------------------------------------------------------
// "Far" candidates (outside the shared-memory window) are read from global
// memory.  With one row per lane every load instruction touches 32 different
// 128-byte lines (32 L1 wavefronts); the row-major layout below puts the NW
// words of a row on NW adjacent lanes, so an instruction covers 32/NW rows and
// only 32/NW (+ straddle) lines: 4-6x fewer L1 wavefronts per candidate.
// One candidate occupies the whole warp; the sum is over all 32 lanes.
// ---------------------------------------------------------------------------
template <typename T, int W, bool SKIP>
struct FarL {
  static constexpr int NW = W * (int)sizeof(T) / 4;  // words (= lanes) per row
  static constexpr int RPI = 32 / NW;                // rows per instruction
  static constexpr int ROWS = SKIP ? W / 2 : W;
  static constexpr int IT = ROWS / RPI;              // iterations
  static constexpr int RSTEP = SKIP ? 2 : 1;
};

template <typename T, int W, bool SKIP>
__device__ __forceinline__ void far_load_src(const T *src, int stride, int lane, uint32_t (&sf)[FarL<T, W, SKIP>::IT]) {
  using F = FarL<T, W, SKIP>;
  const int j = lane % F::NW, rr = lane / F::NW;
#pragma unroll
  for (int it = 0; it < F::IT; it++)
    sf[it] = __ldg(reinterpret_cast<const uint32_t *>(src + (it * F::RPI + rr) * F::RSTEP * stride) + j);
}

// Partial (per-lane) SAD of a far candidate, given as a byte offset from a per-lane base pointer
// (base = ref + this lane's row offset + word column), so the per-candidate address
// arithmetic is one 64-bit add.
template <typename T, int W, bool SKIP>
__device__ __forceinline__ unsigned far_partial_off(const unsigned char *lane_base, int off, int stride,
                                                    const uint32_t (&sf)[FarL<T, W, SKIP>::IT], unsigned sa = 0) {
  using F = FarL<T, W, SKIP>;
  const uintptr_t a = reinterpret_cast<uintptr_t>(lane_base + off);
  const uint32_t *wp = reinterpret_cast<const uint32_t *>(a & ~(uintptr_t)3);
  const unsigned sh = (unsigned)(a & 3) * 8;
  const int step_words = F::RPI * F::RSTEP * stride * (int)sizeof(T) / 4;
  uint32_t w0[F::IT], w1[F::IT];
#pragma unroll
  for (int it = 0; it < F::IT; it++) {
    w0[it] = __ldg(wp + it * step_words);
    w1[it] = __ldg(wp + it * step_words + 1);
  }
  if (sizeof(T) != 1) {  // a + b - 2 min(a, b), as in sad_partial_win
    unsigned accb = 0, accm = 0;
#pragma unroll
    for (int it = 0; it < F::IT; it++) {
      const unsigned x = __funnelshift_r(w0[it], w1[it], sh);
      accb = __dp2a_lo(x, 0x0101u, accb);
      accm = __dp2a_lo(__vminu2(x, sf[it]), 0x0101u, accm);
    }
    return sa + accb - 2 * accm;
  }
  unsigned s = 0;
#pragma unroll
  for (int it = 0; it < F::IT; it++) s = __vsadu4(__funnelshift_r(w0[it], w1[it], sh), sf[it]) + s;
  return s;
}

// ---------------------------------------------------------------------------
// Variance (aom_dsp/variance.c:56-72,141-148; hbd :342-429).  a - b, W x W.
// Lane = column (W == 32) or (row half, column) (W == 16).
// ---------------------------------------------------------------------------
__device__ __forceinline__ unsigned var_finish(int sum, unsigned long long sse, int W, int hbd_shift,
                                               unsigned *sse_out) {
  if (hbd_shift == 0) {
    const unsigned sse32 = (unsigned)sse;
    *sse_out = sse32;
    return sse32 - (unsigned)(((long long)sum * sum) / (W * W));
  }
  const int sh = hbd_shift;
  const unsigned sse32 = (unsigned)((sse + ((1ull << (2 * sh)) >> 1)) >> (2 * sh));
  const int s = (int)(((long long)sum + ((1 << sh) >> 1)) >> sh);
  *sse_out = sse32;
  const long long var = (long long)sse32 - (((long long)s * s) / (W * W));
  return var >= 0 ? (unsigned)var : 0u;
}

template <typename T, int W>
__device__ __forceinline__ unsigned variance(const T *a, int as, const T *b, int bs, int hbd_shift, unsigned *sse_out) {
  const int lane = lane_id();
  constexpr int RP = 32 / W;  // rows per iteration
  const int col = lane % W, r0 = lane / W;
  int sum = 0;
  unsigned sse = 0;
#pragma unroll 8
  for (int i = r0; i < W; i += RP) {
    const int d = (int)__ldg(a + i * as + col) - (int)__ldg(b + i * bs + col);
    sum += d;
    sse += (unsigned)(d * d);
  }
  const unsigned long long sse64 = warp_sum_pair(sum, sse);
  return var_finish(sum, sse64, W, hbd_shift, sse_out);
}

template <typename T, int W>
__device__ __forceinline__ unsigned bilinear_err(const Search<T> &S_in, int r8, int c8, int mode = 1);

// get_mvpred_var_cost (mcomp.c:645-664): vf(src, ref@mv) + L1 cost.
// For 16-bit samples the variance at a full-pel MV is the sub-pel error routine at phase (0, 0)
// (both taps collapse to a copy): same packed arithmetic, and the reference block comes from the
// shared-memory window whenever the MV lies inside it instead of from global memory.
template <typename T, int W>
__device__ __forceinline__ int var_cost(const Search<T> &S, int r, int c) {
  // vf(src, ref): the difference is src - ref, and the high-bitdepth rounding of the sum
  // (ROUND_POWER_OF_TWO of a signed value) is not symmetric under negation -> mode 3
  return (int)bilinear_err<T, W>(S, r * 8, c * 8, 3) + sse_cost(S, r * 8, c * 8);
}

// ---------------------------------------------------------------------------
// diamond_search_sad (mcomp.c:1299-1416).  Kept out of line (one copy per
// layout) so the kernel stays inside the instruction cache.
//
// The reference walks the sites of a stage in index order with a running
// threshold: accept iff sad + cost < bestsad (strict).  Because cost >= 0 the
// inner "sad < bestsad" pre-test is redundant, so the stage result is the
// arg-min of (sad + cost) with ties going to the lowest site index, accepted
// iff it beats the incumbent.  That is evaluated here as a warp min-reduction
// over keys (total << 4 | site index): bit-exact, and without any sequential
// per-candidate code.
//
// Row-sum bound (16x16 search, S.rs set): with S_k the sum of source row k and R_k(mv) the sum of the same W
// reference samples at the candidate, sum_k |S_k - R_k(mv)| <= SAD(mv) over the rows k the SAD reads (triangle
// inequality), and sad_post is monotone.  A site with sad_post(bound) + cost >= bestsad can therefore never be
// accepted, nor be the stage's winning key (a winner beats the stage-start incumbent): it is skipped, exactly as
// the cost pruning skips sites with cost >= bestsad.  The 16x16 search starts at the rounding of its 32x32 block's
// MV, usually at or next to the match, so most later sites fall to the bound.  Applied to the far stages, where a
// skipped site saves its L2 loads.  (Measured and rejected: screening the near stages too and packing their
// surviving sites into the passes -- the row-sum loads cost more than the shared-memory passes they save: 4K
// 10-bit 66.0 vs 69.2 frames/s.)
// ---------------------------------------------------------------------------
template <typename T, int W, bool SKIP>
__device__ __forceinline__ unsigned diamond_search(const Search<T> &S_in, MV2 start, int search_step, int *num00,
                                                MV2 *best_out) {
  using L = SadL<T, W, SKIP>;
  constexpr int PU = (W == 32) ? 2 : (L::MAXP < TF_PU16 ? L::MAXP : TF_PU16);  // passes whose loads are issued back to back
  const Search<T> S = S_in;
  const int lane = lane_id();
  const int grp = lane / L::LPC, row = (lane % L::LPC) * L::RSTEP;
  const unsigned char *safe = reinterpret_cast<const unsigned char *>(S.src);
  uint32_t sw[L::NW];
  sad_load_src<T, W, SKIP>(S.src, S.stride, sw);
  uint32_t sf[FarL<T, W, SKIP>::IT];
  far_load_src<T, W, SKIP>(S.src, S.stride, lane, sf);
  unsigned sa_near = 0, sa_far = 0;  // sums of this lane's source samples in the two layouts (16-bit SAD)
  if (sizeof(T) != 1) {
#pragma unroll
    for (int j = 0; j < L::NW; j++) sa_near = __dp2a_lo(sw[j], 0x0101u, sa_near);
#pragma unroll
    for (int it = 0; it < FarL<T, W, SKIP>::IT; it++) sa_far = __dp2a_lo(sf[it], 0x0101u, sa_far);
  }
  // the bound serves the skip-row SAD only: the full-row pass (small frames, or after a failed skip-row audit)
  // runs without it
  constexpr bool RSB = W == 16 && SKIP;
  constexpr int NPK = RSB ? L::ROWS / 2 : 1;
  const bool use_rs = RSB && S.rs != nullptr;
  unsigned srow = sa_near;  // sum of this lane's source row: lanes 0 .. ROWS - 1 hold S_k of the SAD rows in order
  if (RSB && sizeof(T) == 1) {
#pragma unroll
    for (int j = 0; j < L::NW; j++) srow = __vsadu4(sw[j], 0u) + srow;
  }
  uint32_t spk[NPK];  // S_k two per register, gathered per far stage (warp-uniform) rather than held: registers
  auto rs_gather = [&]() {
#pragma unroll
    for (int j = 0; j < NPK; j++) spk[j] = __shfl_sync(FULL, srow, 2 * j) | (__shfl_sync(FULL, srow, 2 * j + 1) << 16);
  };
  // sad_post of the row-sum bound of the site (r, c) after rs_gather(); only for sites inside the MV limits
  auto rs_bound = [&](int r, int c) -> unsigned {
    const uint16_t *p = S.rs + r * S.stride + c;
    const int step = L::RSTEP * S.stride;
    unsigned b = 0;
#pragma unroll
    for (int j = 0; j < NPK; j++)
      b = __vsadu2((unsigned)__ldg(p + 2 * j * step) | ((unsigned)__ldg(p + (2 * j + 1) * step) << 16), spk[j]) + b;
    return sad_post<SKIP>(b, S.hbd_shift);
  };
  unsigned npruned = 0;  // sites skipped by the bound (instrumentation)
  // this lane's row / word position inside a far candidate (row-major layout)
  const unsigned char *far_base = reinterpret_cast<const unsigned char *>(
      S.ref + (lane / FarL<T, W, SKIP>::NW) * FarL<T, W, SKIP>::RSTEP * S.stride) + 4 * (lane % FarL<T, W, SKIP>::NW);
  start.col = iclamp(start.col, S.lim.col_min, S.lim.col_max);
  start.row = iclamp(start.row, S.lim.row_min, S.lim.row_max);
  const int tot_steps = 15 - search_step;
  int n00 = 0;
  MV2 best = start;
  unsigned bestsad = sad_single<T, W, SKIP>(S, start.row, start.col, lane, sw) + sad_cost(S, start.row, start.col);
  int is_off_center = 0;
  unsigned ncand = 1;  // candidates whose samples were read (instrumentation)
  int next_step_size = tot_steps > 2 ? c_sites.radius[tot_steps - 2] : 1;
  for (int step = tot_steps - 1; step >= 0; --step) {
    if (step > 0) next_step_size = c_sites.radius[step - 1];
    const int nsites = c_sites.n[step];
    const int rad = c_sites.radius[step];
    // all_in tests only the four axis sites (mcomp.c:1339-1344)
    const bool all_in = (best.row - rad >= S.lim.row_min) && (best.row + rad <= S.lim.row_max) &&
                        (best.col - rad >= S.lim.col_min) && (best.col + rad <= S.lim.col_max);
    unsigned mykey = 0xffffffffu;
    // lane i holds the offset of site i of this stage (one constant load per stage; the per-pass
    // lookups are shuffles instead of lane-divergent constant loads)
    // (16x16 search only: the 32x32 search has two lane groups and no registers to spare)
    constexpr bool SHFL_SITES = (W == 16);
    const int site_r = (SHFL_SITES && lane <= nsites) ? (int)c_sites.r[step][lane] : 0;
    const int site_c = (SHFL_SITES && lane <= nsites) ? (int)c_sites.c[step][lane] : 0;
    auto site_row = [&](int i) { return SHFL_SITES ? __shfl_sync(FULL, site_r, i) : (int)c_sites.r[step][i]; };
    auto site_col = [&](int i) { return SHFL_SITES ? __shfl_sync(FULL, site_c, i) : (int)c_sites.c[step][i]; };
    if (window_covers(S, best.row, best.col, rad)) {
      const unsigned worg = (unsigned)__cvta_generic_to_shared(S.win) +
                            (unsigned)((S.wR - S.wr) * S.wpitch + (S.wR - S.wc) * (int)sizeof(T) + S.wshift);
#pragma unroll 1
      for (int p0 = 0; p0 * L::CPP < nsites; p0 += PU) {
        unsigned part[PU];
        int cost[PU];
        bool ok[PU];
#pragma unroll
        for (int u = 0; u < PU; u++) {  // independent loads + partial SADs
          if (u > 0 && (p0 + u) * L::CPP >= nsites) break;  // 8-site stages need fewer passes (uniform)
          const int idx = 1 + (p0 + u) * L::CPP + grp;
          const bool live = idx <= nsites;
          const int sidx = live ? idx : 0;  // site 0 = the centre: always inside the window
          const int my_r = best.row + site_row(sidx);
          const int my_c = best.col + site_col(sidx);
          cost[u] = sad_cost(S, my_r, my_c);
          // exact pruning: a site is accepted only if sad + cost < bestsad and sad >= 0
          ok[u] = live & (all_in | in_range(S.lim, my_r, my_c)) & ((unsigned)cost[u] < bestsad);
          part[u] = sad_partial_win<T, W, SKIP>(worg, S.wpitch, my_r, my_c, row, sw, sa_near);
        }
        ncand += imin(PU * L::CPP, nsites - p0 * L::CPP);
#pragma unroll
        for (int u = 0; u < PU; u++) {
          if (u > 0 && (p0 + u) * L::CPP >= nsites) break;
          const unsigned tot = sad_post<SKIP>(seg_reduce_u32<L::LPC>(part[u]), S.hbd_shift) + (unsigned)cost[u];
          const unsigned key = (tot << 4) | (unsigned)(1 + (p0 + u) * L::CPP + grp);
          mykey = min(mykey, ok[u] ? key : 0xffffffffu);
        }
      }
      mykey = group_min_u32<L::LPC>(mykey);
    } else {
      // far stage: one candidate per warp pass, row-major lanes, 4 candidates in flight.
      // Lane l < nsites prepares site l + 1 once (position, cost, validity, byte offset); the
      // evaluation loop only broadcasts.
      const int mine = ((lane >> 4) & 1) * 2 + ((lane >> 3) & 1);  // candidate this lane owns after reduce4
      const int sidx = lane < nsites ? lane + 1 : 0;
      const int sr = best.row + site_row(sidx), sc = best.col + site_col(sidx);
      const unsigned scost = (unsigned)sad_cost(S, sr, sc);
      // exact pruning: sad + cost < bestsad is impossible once cost >= bestsad
      bool sok = (lane < nsites) & (all_in | in_range(S.lim, sr, sc)) & (scost < bestsad);
      if (use_rs) {
        const unsigned cmask = __ballot_sync(FULL, sok);
        rs_gather();
        if (sok) sok = rs_bound(sr, sc) + scost < bestsad;
        npruned += __popc(cmask & ~__ballot_sync(FULL, sok));
      }
      const int soff = (sr * S.stride + sc) * (int)sizeof(T);
      const unsigned okmask = __ballot_sync(FULL, sok);
      // (Measured and rejected: reading a quarter of a far candidate's rows first and dropping it when that
      // part alone reaches the incumbent -- exact, but the 32x32 search walks its far stages against the poor
      // incumbent of a predicted start, few candidates die early, and the second dependent load round trip
      // lengthens the chain: 45.9 vs 51.0 frames/s.)
      ncand += __popc(okmask);
#pragma unroll 1
      for (int i0 = 0; i0 < nsites; i0 += 4) {
        if (((okmask >> i0) & 15u) == 0) continue;
        unsigned part[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
          const int off = __shfl_sync(FULL, soff, i0 + u);
          part[u] = ((okmask >> (i0 + u)) & 1u) ? far_partial_off<T, W, SKIP>(far_base, off, S.stride, sf, sa_far) : 0u;
        }
        const unsigned tot4 = reduce4_u32(part, lane);
        const unsigned my_cost = __shfl_sync(FULL, scost, i0 + mine);
        const unsigned tot = sad_post<SKIP>(tot4, S.hbd_shift) + my_cost;
        mykey = min(mykey, ((okmask >> (i0 + mine)) & 1u) ? ((tot << 4) | (unsigned)(i0 + mine + 1)) : 0xffffffffu);
      }
      mykey = min(mykey, __shfl_xor_sync(FULL, mykey, 8));
      mykey = min(mykey, __shfl_xor_sync(FULL, mykey, 16));
      // (Measured and rejected in round 2, same box A/B at 4K 10-bit: REDUX.SUM / REDUX.MIN instead of the shuffle
      // trees 52.25 vs 52.83 frames/s; an L1 prefetch (CCTL.PF1) of every live candidate of the stage before the
      // loop 53.9 vs 56.3; live candidates packed four to a pass instead of fixed groups 55.8 vs 56.3.)
    }
    int best_site = 0;
    if ((mykey >> 4) < bestsad) {
      bestsad = mykey >> 4;
      best_site = (int)(mykey & 15u);
    }
    if (best_site != 0) {
      best.row += site_row(best_site);
      best.col += site_col(best_site);
      is_off_center = 1;
    }
    if (is_off_center == 0) n00++;
    if (best_site == 0) {
      while (next_step_size == c_sites.radius[step] && step > 2) {
        ++n00;
        --step;
        next_step_size = c_sites.radius[step - 1];
      }
    }
  }
  if (S.ctr && lane == 0) {
    atomicAdd(&S.ctr[0], (unsigned long long)ncand * (L::ROWS * W));
    if (use_rs) atomicAdd(&S.ctr[3], (unsigned long long)npruned);
  }
  *num00 = n00;
  *best_out = best;
  return bestsad;
}

// full_pixel_diamond (mcomp.c:1421-1470), cost_list == NULL
template <typename T, int W, bool SKIP>
__device__ int full_pixel_diamond(const Search<T> &S, MV2 start, int step_param, MV2 *best_mv) {
  int n = 0, num00 = 0;
  int bestsme = 0;
  const int further_steps = 15 - 1 - step_param;
  // first pass (pass_n = 0) and the refinement passes share one call site
  bool first = true;
  MV2 memo_mv = { 0x7fff, 0x7fff };
  int memo_sme = 0;
  while (first || n < further_steps) {
    if (!first) {
      ++n;
      if (num00) {
        num00--;
        continue;
      }
    }
    MV2 tmp;
    int nn;
    int thissme = (int)diamond_search<T, W, SKIP>(S, start, step_param + (first ? 0 : n), &nn, &tmp);
    if (thissme < INT_MAX_) {
      // var_cost is a pure function of the MV: passes that end on an MV already scored reuse the value
      if (!first && tmp.row == best_mv->row && tmp.col == best_mv->col) thissme = bestsme;
      else if (!first && tmp.row == memo_mv.row && tmp.col == memo_mv.col) thissme = memo_sme;
      else {
        thissme = var_cost<T, W>(S, tmp.row, tmp.col);
        memo_mv = tmp;
        memo_sme = thissme;
      }
    }
    if (first) {
      n = nn;
      bestsme = thissme;
      *best_mv = tmp;
      first = false;
    } else {
      num00 = nn;
      if (thissme < bestsme) {
        bestsme = thissme;
        *best_mv = tmp;
      }
    }
  }
  return bestsme;
}

// exhaustive_mesh_search (mcomp.c:1474-1543).  The visiting order is the
// reference's (row major; with step == 1 the 4-wide groups and the tail quirk
// that never visits end_col unless the column count is a multiple of 4).
// update_mvs_and_sad (:839-858) is a running strict minimum of sad + cost in
// visiting order = arg-min with ties to the earliest visit, so every lane
// group keeps the best key (total << 32 | visit index) of the candidates it
// evaluated and one warp min-reduction at the end picks the winner.
template <typename T, int W, bool SKIP>
__device__ __forceinline__ int mesh_search(const Search<T> &S_in, MV2 start, int range, int step, MV2 *best_out) {
  using L = SadL<T, W, SKIP>;
  constexpr int PU = 2;
  const Search<T> S = S_in;
  const int lane = lane_id();
  const int grp = lane / L::LPC, row = (lane % L::LPC) * L::RSTEP;
  const unsigned char *safe = reinterpret_cast<const unsigned char *>(S.src);
  uint32_t sw[L::NW];
  sad_load_src<T, W, SKIP>(S.src, S.stride, sw);
  start.col = iclamp(start.col, S.lim.col_min, S.lim.col_max);
  start.row = iclamp(start.row, S.lim.row_min, S.lim.row_max);
  MV2 best = start;
  unsigned best_sad = sad_single<T, W, SKIP>(S, start.row, start.col, lane, sw) + sad_cost(S, start.row, start.col);
  const int start_row = imax(-range, S.lim.row_min - start.row);
  const int start_col = imax(-range, S.lim.col_min - start.col);
  const int end_row = imin(range, S.lim.row_max - start.row);
  const int end_col = imin(range, S.lim.col_max - start.col);
  *best_out = best;
  if (end_row < start_row || end_col < start_col) return (int)best_sad;
  const int n_rows = (end_row - start_row) / step + 1;
  int n_cols;
  if (step > 1) {
    n_cols = (end_col - start_col) / step + 1;
  } else {
    const int ncols = end_col - start_col + 1;
    n_cols = (ncols % 4 == 0) ? ncols : ncols - 1;
  }
  const int total = n_rows * n_cols;
  const SadSrc Q = sad_src(S, window_covers(S, start.row, start.col, range));
  unsigned long long mykey = ~0ull;
#pragma unroll 1
  for (int q0 = 0; q0 < total; q0 += L::CPP * PU) {
    unsigned part[PU];
    int cost[PU];
#pragma unroll
    for (int u = 0; u < PU; u++) {
      const int q = q0 + u * L::CPP + grp;
      const bool valid = q < total;
      const int qq = valid ? q : 0;
      const int ri = qq / n_cols, ci = qq - ri * n_cols;
      const int my_r = start.row + start_row + ri * step, my_c = start.col + start_col + ci * step;
      cost[u] = sad_cost(S, my_r, my_c);
      part[u] = sad_partial<T, W, SKIP>(Q, safe, my_r, my_c, row, valid && (unsigned)cost[u] < best_sad, sw);
    }
#pragma unroll
    for (int u = 0; u < PU; u++) {
      const int q = q0 + u * L::CPP + grp;
      const unsigned tot = sad_post<SKIP>(seg_reduce_u32<L::LPC>(part[u]), S.hbd_shift) + (unsigned)cost[u];
      const unsigned long long key = ((unsigned long long)tot << 32) | (unsigned)q;
      mykey = (q < total && (unsigned)cost[u] < best_sad && key < mykey) ? key : mykey;
    }
  }
#pragma unroll
  for (int o = L::LPC; o < 32; o <<= 1) {
    const unsigned long long other = __shfl_xor_sync(FULL, mykey, o);
    mykey = other < mykey ? other : mykey;
  }
  if (S.ctr && lane == 0) atomicAdd(&S.ctr[0], (unsigned long long)(total + 1) * (L::ROWS * W));
  if ((unsigned)(mykey >> 32) < best_sad) {
    best_sad = (unsigned)(mykey >> 32);
    const int q = (int)(mykey & 0xffffffffull);
    const int ri = q / n_cols;
    best.row = start.row + start_row + ri * step;
    best.col = start.col + start_col + (q - ri * n_cols) * step;
  }
  *best_out = best;
  return (int)best_sad;
}

// full_pixel_exhaustive (mcomp.c:1547-1617)
template <typename T, int W, bool SKIP>
__device__ int full_pixel_exhaustive(Search<T> &S, const KParams &P, MV2 start, MV2 *best_mv, unsigned char *winbuf) {
  int interval = P.mesh[0][1], range = P.mesh[0][0];
  *best_mv = start;
  if (range < 7 || range > 256 || interval < 1 || interval > range) return INT_MAX_;
  const int baseline_interval_divisor = range / interval;
  range = imax(range, (5 * imax(iabs(best_mv->row), iabs(best_mv->col))) / 4);
  range = imin(range, 256);
  interval = imax(interval, range / baseline_interval_divisor);
  int bestsme = 0;
  for (int i = 0; i < 4; ++i) {  // pass 0, then patterns 1.. until an interval-1 pattern has run
    if (i > 0) {
      range = P.mesh[i][0];
      interval = P.mesh[i][1];
    }
    MV2 nb;
    if (!window_covers(S, best_mv->row, best_mv->col, range) && range <= WinCfg<T, W>::R)
      window_load<T, W>(S, winbuf, best_mv->row, best_mv->col);
    bestsme = mesh_search<T, W, SKIP>(S, *best_mv, range, interval, &nb);
    *best_mv = nb;
    if (i == 0 && !(interval > 1 && range > 7)) break;
    if (i > 0 && P.mesh[i][1] == 1) break;
  }
  if (bestsme < INT_MAX_) bestsme = var_cost<T, W>(S, best_mv->row, best_mv->col);
  return bestsme;
}

// av1_full_pixel_search (mcomp.c:1693-1832), NSTEP, run_mesh_search = 1.
// Returns 1 when the skip-row result must be discarded and the search redone
// with full SAD (mcomp.c:1777-1810).
template <typename T, int W, bool SKIP>
__device__ __forceinline__ int full_pixel_search_pass(Search<T> &S, const KParams &P, MV2 start, MV2 *best_mv,
                                                   unsigned char *winbuf) {
  int run_mesh = 1;
  int var = full_pixel_diamond<T, W, SKIP>(S, start, P.step_param, best_mv);
  int prune = 0, thr = 4;
  if (P.prune_level == 2) prune = 1;
  if (P.prune_level == 1) {
    prune = (P.q_factor <= 20) ? 0 : 1;
    thr = 2;
  }
  if (prune) {
    const int d = imax(iabs(start.row - best_mv->row), iabs(start.col - best_mv->col));
    if (d <= thr) run_mesh = 0;
  }
  if (SKIP) {
    // sdf and sdsf at best_mv: one full-row SAD pass (one block row per lane, the window when best_mv lies
    // inside it); the skip-row SAD is the sum over the even rows of the same pass
    using LF = SadL<T, W, false>;
    const int lane = lane_id();
    const int row = lane % LF::LPC;
    uint32_t swf[LF::NW];
    sad_load_src<T, W, false>(S.src, S.stride, swf);
    const SadSrc Q = sad_src(S, window_covers(S, best_mv->row, best_mv->col, 0));
    const unsigned part = sad_partial<T, W, false>(Q, reinterpret_cast<const unsigned char *>(S.src), best_mv->row,
                                                   best_mv->col, row, true, swf);
    const unsigned s_all = seg_reduce_u32<LF::LPC>(part);
    const unsigned s_even = seg_reduce_u32<LF::LPC>((row & 1) ? 0u : part);
    const int sad = (int)(s_all >> S.hbd_shift);
    const int skip_sad = (int)((2 * s_even) >> S.hbd_shift);
    const int kSADThresh = W * W / 16;
    if (sad > kSADThresh && iabs(skip_sad - sad) * 10 >= imax(sad, 1) * 9) return 1;
  }
  if (run_mesh) {
    MV2 tmp;
    const int var_ex = full_pixel_exhaustive<T, W, SKIP>(S, P, *best_mv, &tmp, winbuf);
    if (var_ex < var) {
      var = var_ex;
      *best_mv = tmp;
    }
  }
  return 0;
}

template <typename T, int W>
__device__ void full_pixel_search(Search<T> &S, const KParams &P, MV2 start, MV2 *best_mv, unsigned char *winbuf) {
  const int wr = iclamp(start.row, S.lim.row_min, S.lim.row_max);
  const int wc = iclamp(start.col, S.lim.col_min, S.lim.col_max);
  window_load<T, W>(S, winbuf, wr, wc);
  // The window stays valid for the bilinear sub-pel search that follows (its candidates surround
  // best_mv, normally inside the window); SUBPEL_TREE reuses the buffer as 8-tap scratch instead.
  const bool keep = P.subpel_method != 0;
  if (P.use_skip) {
    if (!full_pixel_search_pass<T, W, true>(S, P, start, best_mv, winbuf)) {
      if (!keep) S.win = nullptr;
      return;
    }
    if (S.wr != wr || S.wc != wc) window_load<T, W>(S, winbuf, wr, wc);
  }
  full_pixel_search_pass<T, W, false>(S, P, start, best_mv, winbuf);
  if (!keep) S.win = nullptr;
}

// ---------------------------------------------------------------------------
// Sub-pel search
// ---------------------------------------------------------------------------
// aom_sub_pixel_variance (aom_dsp/variance.c:91-139,150-163; hbd :478-560):
// 2-tap bilinear over (W+1) x (W+1) samples then variance(filtered, src).
// mode 1: sub-pel candidate (difference = filtered ref - src, as vf(pred, src) in mcomp.c:2385-2425);
// mode 2: full-pel variance vf(ref, src); mode 3: full-pel variance vf(src, ref) (difference negated).
// Modes 2 and 3 count as variance work in the instrumentation.
template <typename T, int W>
__device__ __forceinline__ unsigned bilinear_err(const Search<T> &S_in, int r8, int c8, int mode) {
  const Search<T> S = S_in;
  const int lane = lane_id();
  const int fr = r8 >> 3, fc = c8 >> 3;
  const int xo = c8 & 7, yo = r8 & 7;
  // Two samples per 32-bit register (16-bit halves; 8-bit samples are widened on load).  The taps
  // {128 - 16k, 16k} share the factor 16, so
  // ROUND_POWER_OF_TWO(a0 * (128 - 16k) + a1 * 16k, 7) == (a0 * (8 - k) + a1 * k + 4) >> 3 exactly,
  // and with samples <= 4095 every term stays below 2^16: both halves of a register go through one
  // IMAD without carrying into each other.  Lane = (row band, column pair).
  constexpr int ES = (int)sizeof(T);
  constexpr int PAIRS = W / 2;          // lanes per block row
  constexpr int BANDS = 32 / PAIRS;     // 2 (W = 32) or 4 (W = 16)
  constexpr int BROWS = W / BANDS;      // 16 or 4 rows per band
  constexpr int CH = BROWS < 8 ? BROWS : 8;
  const int j = lane % PAIRS, rbeg = (lane / PAIRS) * BROWS;
  // (fr, fc) and (fr + 1, fc + 1) inside the search window -> read it from shared memory
  const SadSrc Q = sad_src(S, window_covers(S, fr, fc, 1) && S.wr - fr < S.wR && S.wc - fc < S.wR);
  const uintptr_t a = reinterpret_cast<uintptr_t>(Q.base + (fr + rbeg) * Q.pitchB + (fc + 2 * j) * ES);
  const unsigned char *wb = reinterpret_cast<const unsigned char *>(a & ~(uintptr_t)3);
  const unsigned sh = (unsigned)(a & 3) * 8;  // row pitches are multiples of 4 bytes: same for every row
  const int sstep = S.stride / 2;             // source row step in pairs
  const unsigned m0 = 8 - xo, m1 = xo, n0 = 8 - yo, n1 = yo;
  constexpr unsigned RND = 0x00040004u, MSK = 0x1fff1fffu;
  auto hrow = [&](uint32_t w0, uint32_t w1) -> unsigned {
    unsigned A, B;  // samples (x, x + 1) and (x + 1, x + 2)
    if (ES == 2) {
      A = __funnelshift_rc(w0, w1, sh);
      B = __funnelshift_rc(w0, w1, sh + 16);
    } else {
      const unsigned x = __funnelshift_r(w0, w1, sh);  // bytes x .. x + 3
      A = __byte_perm(x, 0, 0x4140);
      B = __byte_perm(x, 0, 0x4241);
    }
    return ((A * m0 + (B * m1 + RND)) >> 3) & MSK;
  };
  auto src_pair = [&](int r) -> unsigned {
    if (ES == 2) return __ldg(reinterpret_cast<const uint32_t *>(S.src + rbeg * S.stride + 2 * j) + r * sstep);
    const unsigned s = __ldg(reinterpret_cast<const uint16_t *>(S.src + rbeg * S.stride + 2 * j) + r * sstep);
    return __byte_perm(s, 0, 0x4140);
  };
  unsigned hprev;
  {
    const uint32_t *wp = reinterpret_cast<const uint32_t *>(wb);
    hprev = hrow(wp[0], wp[1]);
  }
  unsigned sumv = 0, sums = 0, accl = 0, acch = 0;
#pragma unroll 1
  for (int t0 = 0; t0 < BROWS; t0 += CH) {
    uint32_t w0[CH], w1[CH], sv[CH];
#pragma unroll
    for (int k = 0; k < CH; k++) {  // all loads of a chunk are issued before use
      const uint32_t *wp = reinterpret_cast<const uint32_t *>(wb + (t0 + k + 1) * Q.pitchB);
      w0[k] = wp[0];
      w1[k] = wp[1];
    }
#pragma unroll
    for (int k = 0; k < CH; k++) sv[k] = src_pair(t0 + k);
#pragma unroll
    for (int k = 0; k < CH; k++) {
      const unsigned hn = hrow(w0[k], w1[k]);
      const unsigned v = ((hprev * n0 + (hn * n1 + RND)) >> 3) & MSK;
      hprev = hn;
      sumv = __dp2a_lo(v, 0x0101u, sumv);
      sums = __dp2a_lo(sv[k], 0x0101u, sums);
      const unsigned md = __vmaxu2(v, sv[k]) - __vminu2(v, sv[k]);  // |v - s| per half
      const unsigned pb = __byte_perm(md, 0, 0x3120);                // (d0.lo, d1.lo, d0.hi, d1.hi)
      accl = __dp2a_lo(md, pb, accl);                                // sum d * (d & 255)
      if (ES == 2) acch = __dp2a_hi(md, pb, acch);                   // sum d * (d >> 8)
    }
  }
  if (S.ctr && lane == 0) atomicAdd(&S.ctr[mode == 1 ? 1 : 2], (unsigned long long)(W * W));
  int sum = mode == 3 ? (int)sums - (int)sumv : (int)sumv - (int)sums;
  const unsigned long long sse64 = warp_sum_pair(sum, accl + (acch << 8));
  unsigned sse_out;
  return var_finish(sum, sse64, W, S.hbd_shift, &sse_out);
}

// ---------------------------------------------------------------------------
// Sub-pel error out of shared memory only.  subpel_search() makes sure the search window covers every
// candidate of the sub-pel stage (all lie within two full-pel steps of its start) and the source block is
// staged as a tile, so these routines use ld.shared with 32-bit addresses and compile-time row pitches (no
// generic loads, no 64-bit address arithmetic per row).  Same taps and rounding as bilinear_err; the error
// terms use a biased difference: d' = v + 4096 - s is positive in both halves of the register, so one IADD3
// replaces max / min / subtract, one IDP.2A sums it, and
//   sum(d) = sum(d') - 4096 n,   sum(d^2) = sum(d'^2) - 8192 sum(d') + n 2^24   (exact; evaluated mod 2^32,
// the true per-lane value is below 2^32).
// ---------------------------------------------------------------------------
template <typename T, int W>
__device__ __forceinline__ unsigned win_origin(const Search<T> &S) {  // shared address of MV (0, 0), row 0
  return (unsigned)__cvta_generic_to_shared(S.win) +
         (unsigned)((S.wR - S.wr) * WinCfg<T, W>::PITCH + (S.wR - S.wc) * (int)sizeof(T) + S.wshift);
}
template <typename T, int W>
__device__ __forceinline__ unsigned subpel_err_win(const Search<T> &S_in, int r8, int c8, int mode) {
  const Search<T> S = S_in;
  const int lane = lane_id();
  const int fr = r8 >> 3, fc = c8 >> 3;
  const int xo = c8 & 7, yo = r8 & 7;
  constexpr int ES = (int)sizeof(T);
  constexpr int WP = WinCfg<T, W>::PITCH, SP = SrcTile<T, W>::PITCH;
  constexpr int PAIRS = W / 2, BANDS = 32 / PAIRS, BROWS = W / BANDS;
  constexpr int CH = BROWS < 8 ? BROWS : 8;
  const int j = lane % PAIRS, rbeg = (lane / PAIRS) * BROWS;
  const unsigned a = win_origin<T, W>(S) + (unsigned)((fr + rbeg) * WP + (fc + 2 * j) * ES);
  const unsigned wa = a & ~3u, sh = (a & 3u) * 8;
  const unsigned sa = S.srcs + (unsigned)(rbeg * SP + 2 * j * ES);
  const unsigned m0 = 8 - xo, m1 = xo, n0 = 8 - yo, n1 = yo;
  constexpr unsigned RND = 0x00040004u, MSK = 0x1fff1fffu, BIAS = 0x10001000u;
  auto hrow = [&](uint32_t w0, uint32_t w1) -> unsigned {
    unsigned A, B;
    if (ES == 2) {
      A = __funnelshift_rc(w0, w1, sh);
      B = __funnelshift_rc(w0, w1, sh + 16);
    } else {
      const unsigned x = __funnelshift_r(w0, w1, sh);
      A = __byte_perm(x, 0, 0x4140);
      B = __byte_perm(x, 0, 0x4241);
    }
    return ((A * m0 + (B * m1 + RND)) >> 3) & MSK;
  };
  unsigned hprev = hrow(lds_u32(wa), lds_u32(wa + 4));
  unsigned accs = 0, accl = 0, acch = 0;
#pragma unroll 1
  for (int t0 = 0; t0 < BROWS; t0 += CH) {
    uint32_t w0[CH], w1[CH], sv[CH];
    const unsigned wb = wa + (unsigned)((t0 + 1) * WP), sb = sa + (unsigned)(t0 * SP);
#pragma unroll
    for (int k = 0; k < CH; k++) {
      w0[k] = lds_u32(wb + k * WP);
      w1[k] = lds_u32(wb + k * WP + 4);
    }
#pragma unroll
    for (int k = 0; k < CH; k++) sv[k] = ES == 2 ? lds_u32(sb + k * SP) : __byte_perm(lds_u16(sb + k * SP), 0, 0x4140);
#pragma unroll
    for (int k = 0; k < CH; k++) {
      const unsigned hn = hrow(w0[k], w1[k]);
      const unsigned v = ((hprev * n0 + (hn * n1 + RND)) >> 3) & MSK;
      hprev = hn;
      const unsigned dp = v + BIAS - sv[k];
      const unsigned pb = __byte_perm(dp, 0, 0x3120);
      accs = __dp2a_lo(dp, 0x0101u, accs);
      accl = __dp2a_lo(dp, pb, accl);
      acch = __dp2a_hi(dp, pb, acch);
    }
  }
  if (S.ctr && lane == 0) atomicAdd(&S.ctr[mode == 1 ? 1 : 2], (unsigned long long)(W * W));
  constexpr int NL = BROWS * 2;  // samples per lane
  const int sumd = (int)accs - NL * 4096;
  const unsigned sse = accl + (acch << 8) - (accs << 13) + (unsigned)NL * (1u << 24);
  int sum = mode == 3 ? -sumd : sumd;
  const unsigned long long sse64 = warp_sum_pair(sum, sse);
  unsigned sse_out;
  return var_finish(sum, sse64, W, S.hbd_shift, &sse_out);
}
// The four first-level candidates of a sub-pel round (left, right, up, down of (tr, tc) at distance hstep;
// first_level_check, mcomp.c:2503-2541) evaluated in one pass: their errors do not depend on the incumbent, so the
// reference's sequential comparisons can be replayed on the four results afterwards.  Lane group g = lane / 8
// evaluates candidate g; a lane owns one (W = 16) or two (W = 32) column pairs over all rows, so there is no band
// overhead and one reduction / variance epilogue serves all four.  Candidates whose bit in validmask is clear are
// not read (their group re-reads the centre) and return INT_MAX.
template <typename T, int W>
__device__ __forceinline__ uint4 subpel_err4_win(const Search<T> &S_in, int tr, int tc, int hstep, unsigned validmask) {
  const Search<T> S = S_in;
  constexpr int ES = (int)sizeof(T);
  constexpr int WP = WinCfg<T, W>::PITCH, SP = SrcTile<T, W>::PITCH;
  constexpr int NP = W / 16;
  constexpr int CH = NP == 1 ? 8 : 4;
  const int lane = lane_id(), g = lane >> 3, u = lane & 7;
  const bool valid = (validmask >> g) & 1u;
  int r8 = tr, c8 = tc;
  if (valid) {
    if (g == 0) c8 -= hstep;
    else if (g == 1) c8 += hstep;
    else if (g == 2) r8 -= hstep;
    else r8 += hstep;
  }
  const int fr = r8 >> 3, fc = c8 >> 3;
  const unsigned xo = c8 & 7, yo = r8 & 7;
  const unsigned a = win_origin<T, W>(S) + (unsigned)(fr * WP + (fc + 2 * u) * ES);
  const unsigned wa = a & ~3u, sh = (a & 3u) * 8;  // 16 pairs further on is a multiple of 4 bytes: same shift
  const unsigned sa = S.srcs + (unsigned)(2 * u * ES);
  const unsigned m0 = 8 - xo, m1 = xo, n0 = 8 - yo, n1 = yo;
  constexpr unsigned RND = 0x00040004u, MSK = 0x1fff1fffu, BIAS = 0x10001000u;
  auto hrow = [&](uint32_t w0, uint32_t w1) -> unsigned {
    unsigned A, B;
    if (ES == 2) {
      A = __funnelshift_rc(w0, w1, sh);
      B = __funnelshift_rc(w0, w1, sh + 16);
    } else {
      const unsigned x = __funnelshift_r(w0, w1, sh);
      A = __byte_perm(x, 0, 0x4140);
      B = __byte_perm(x, 0, 0x4241);
    }
    return ((A * m0 + (B * m1 + RND)) >> 3) & MSK;
  };
  unsigned hprev[NP];
#pragma unroll
  for (int p = 0; p < NP; p++) hprev[p] = hrow(lds_u32(wa + p * 16 * ES), lds_u32(wa + p * 16 * ES + 4));
  unsigned accs = 0, accl = 0, acch = 0;
#pragma unroll 1
  for (int t0 = 0; t0 < W; t0 += CH) {
    uint32_t w0[CH][NP], w1[CH][NP], sv[CH][NP];
    const unsigned wb = wa + (unsigned)((t0 + 1) * WP), sb = sa + (unsigned)(t0 * SP);
#pragma unroll
    for (int k = 0; k < CH; k++)
#pragma unroll
      for (int p = 0; p < NP; p++) {
        w0[k][p] = lds_u32(wb + k * WP + p * 16 * ES);
        w1[k][p] = lds_u32(wb + k * WP + p * 16 * ES + 4);
      }
#pragma unroll
    for (int k = 0; k < CH; k++)
#pragma unroll
      for (int p = 0; p < NP; p++)
        sv[k][p] = ES == 2 ? lds_u32(sb + k * SP + p * 16 * ES) : __byte_perm(lds_u16(sb + k * SP + p * 16 * ES), 0, 0x4140);
#pragma unroll
    for (int k = 0; k < CH; k++)
#pragma unroll
      for (int p = 0; p < NP; p++) {
        const unsigned hn = hrow(w0[k][p], w1[k][p]);
        const unsigned v = ((hprev[p] * n0 + (hn * n1 + RND)) >> 3) & MSK;
        hprev[p] = hn;
        const unsigned dp = v + BIAS - sv[k][p];
        const unsigned pb = __byte_perm(dp, 0, 0x3120);
        accs = __dp2a_lo(dp, 0x0101u, accs);
        accl = __dp2a_lo(dp, pb, accl);
        acch = __dp2a_hi(dp, pb, acch);
      }
  }
  if (S.ctr && lane == 0) atomicAdd(&S.ctr[1], (unsigned long long)(__popc(validmask & 15u) * W * W));
  constexpr int NL = W * NP * 2;  // samples per lane
  const int sumd = (int)accs - NL * 4096;
  const unsigned sse = accl + (acch << 8) - (accs << 13) + (unsigned)NL * (1u << 24);
  // (sum, sse) of a candidate = totals over its 8 lanes: |sum| < 2^19 per lane, sse totals < 2^35
  unsigned long long pk = ((unsigned long long)sse << 24) | (unsigned)(sumd + (1 << 19));
#pragma unroll
  for (int o = 4; o > 0; o >>= 1) pk += __shfl_xor_sync(FULL, pk, o);
  const int sum = (int)(pk & 0xffffffu) - (1 << 22);
  unsigned sse_out;
  const unsigned mine = valid ? var_finish(sum, pk >> 24, W, S.hbd_shift, &sse_out) : (unsigned)INT_MAX_;
  uint4 out;
  out.x = __shfl_sync(FULL, mine, 0);
  out.y = __shfl_sync(FULL, mine, 8);
  out.z = __shfl_sync(FULL, mine, 16);
  out.w = __shfl_sync(FULL, mine, 24);
  return out;
}
__device__ __forceinline__ int clip_px(int v, int bd) {
  const int m = (1 << bd) - 1;
  return v < 0 ? 0 : (v > m ? m : v);
}

// aom_upsampled_pred_c (reconinter_enc.c:424-496, hbd :656+) with
// EIGHTTAP_REGULAR through aom_convolve8_{horiz,vert}_c (aom_dsp/aom_convolve.c
// :36-72; pixel-range intermediate), then vf(pred, src) (mcomp.c:2385,2405).
// tmp: warp-private shared scratch of at least (W+7)*W samples of T.
template <typename T, int W>
__device__ __noinline__ unsigned upsampled_err(const Search<T> &S, int r8, int c8, int bd, T *tmp) {
  const int lane = lane_id();
  const int st = S.stride;
  const T *ref = S.ref + (r8 >> 3) * st + (c8 >> 3);
  const int sx = c8 & 7, sy = r8 & 7;
  constexpr int RP = 32 / W;
  const int col = lane % W, r0 = lane / W;
  int sum = 0;
  unsigned sse = 0;
  if (sx && sy) {
    const int16_t *kx = c_k8[sx << 1];
    for (int y = r0; y < W + 7; y += RP) {
      int acc = 0;
#pragma unroll
      for (int t = 0; t < 8; t++) acc += (int)__ldg(ref + (y - 3) * st + col - 3 + t) * kx[t];
      tmp[y * W + col] = (T)clip_px(rpot(acc, 7), bd);
    }
    __syncwarp();
  }
  const int16_t *ky = c_k8[sy << 1];
  const int16_t *kx = c_k8[sx << 1];
  for (int y = r0; y < W; y += RP) {
    int v;
    if (!sx && !sy) {
      v = (int)__ldg(ref + y * st + col);
    } else if (!sy) {
      int acc = 0;
#pragma unroll
      for (int t = 0; t < 8; t++) acc += (int)__ldg(ref + y * st + col - 3 + t) * kx[t];
      v = clip_px(rpot(acc, 7), bd);
    } else if (!sx) {
      int acc = 0;
#pragma unroll
      for (int t = 0; t < 8; t++) acc += (int)__ldg(ref + (y - 3 + t) * st + col) * ky[t];
      v = clip_px(rpot(acc, 7), bd);
    } else {
      int acc = 0;
#pragma unroll
      for (int t = 0; t < 8; t++) acc += (int)tmp[(y + t) * W + col] * ky[t];
      v = clip_px(rpot(acc, 7), bd);
    }
    const int d = v - (int)__ldg(S.src + y * st + col);
    sum += d;
    sse += (unsigned)(d * d);
  }
  __syncwarp();
  if (S.ctr && lane == 0) atomicAdd(&S.ctr[1], (unsigned long long)(W * W));
  const unsigned long long sse64 = warp_sum_pair(sum, sse);
  unsigned sse_out;
  return var_finish(sum, sse64, W, S.hbd_shift, &sse_out);
}

template <typename T, int W>
struct Subpel {
  const Search<T> *S;
  Lim lim;
  unsigned besterr;
  MV2 best;
  int bd;
  T *tmp;
};

// check_better_fast / check_better (mcomp.c:2433-2488), MV_COST_NONE
template <typename T, int W>
__device__ __forceinline__ unsigned check_better(Subpel<T, W> &sp, int r8, int c8, bool accurate, int *is_better) {
  if (!in_range(sp.lim, r8, c8)) return (unsigned)INT_MAX_;
  const unsigned cost = accurate ? upsampled_err<T, W>(*sp.S, r8, c8, sp.bd, sp.tmp) : subpel_err_win<T, W>(*sp.S, r8, c8, 1);
  if (cost < sp.besterr) {
    sp.besterr = cost;
    sp.best.row = r8;
    sp.best.col = c8;
    if (is_better) *is_better |= 1;
  }
  return cost;
}

// first_level_check(_fast) (mcomp.c:2503-2541, 2626-2660)
template <typename T, int W>
__device__ MV2 first_level(Subpel<T, W> &sp, MV2 t, int hstep, bool accurate) {
  unsigned left, right, up, down;
  // (Round 1 kept four short passes for the 32x32 search; with the routines inlined and reading shared memory
  // only, the batched pass is faster there too: 60.4 -> 61.5 frames/s at 4K 10-bit.)
  if (accurate) {
    left = check_better(sp, t.row, t.col - hstep, accurate, nullptr);
    right = check_better(sp, t.row, t.col + hstep, accurate, nullptr);
    up = check_better(sp, t.row - hstep, t.col, accurate, nullptr);
    down = check_better(sp, t.row + hstep, t.col, accurate, nullptr);
  } else {
    // one pass for the four candidates, then check_better's comparisons in the reference's order
    const unsigned vm = (in_range(sp.lim, t.row, t.col - hstep) ? 1u : 0u) | (in_range(sp.lim, t.row, t.col + hstep) ? 2u : 0u) |
                        (in_range(sp.lim, t.row - hstep, t.col) ? 4u : 0u) | (in_range(sp.lim, t.row + hstep, t.col) ? 8u : 0u);
    const uint4 c = subpel_err4_win<T, W>(*sp.S, t.row, t.col, hstep, vm);
    left = c.x, right = c.y, up = c.z, down = c.w;
    const int dr[4] = { 0, 0, -hstep, hstep }, dc[4] = { -hstep, hstep, 0, 0 };
    const unsigned cs[4] = { left, right, up, down };
#pragma unroll
    for (int i = 0; i < 4; i++)
      if (cs[i] < sp.besterr) {  // invalid candidates carry INT_MAX and never win
        sp.besterr = cs[i];
        sp.best.row = t.row + dr[i];
        sp.best.col = t.col + dc[i];
      }
  }
  MV2 diag;
  diag.row = up <= down ? -hstep : hstep;
  diag.col = left <= right ? -hstep : hstep;
  check_better(sp, t.row + diag.row, t.col + diag.col, accurate, nullptr);
  return diag;
}

// second_level_check_fast (mcomp.c:2545-2605)
template <typename T, int W>
__device__ void second_level_fast(Subpel<T, W> &sp, MV2 t, MV2 diag, int hstep) {
  const int tr = t.row, tc = t.col, br = sp.best.row, bc = sp.best.col;
  if (tr != br && tc != bc) {
    check_better(sp, br, bc + diag.col, false, nullptr);
    check_better(sp, br + diag.row, bc, false, nullptr);
  } else if (tr == br && tc != bc) {
    check_better(sp, br + hstep, bc + diag.col, false, nullptr);
    check_better(sp, br - hstep, bc + diag.col, false, nullptr);
    check_better(sp, br - diag.row, bc, false, nullptr);
  } else if (tr != br && tc == bc) {
    check_better(sp, br + diag.row, bc + hstep, false, nullptr);
    check_better(sp, br + diag.row, bc - hstep, false, nullptr);
    check_better(sp, br, bc - diag.col, false, nullptr);
  }
}

// second_level_check_v2 (mcomp.c:2665-2715), subpel_search_type = USE_8_TAPS
template <typename T, int W>
__device__ void second_level_v2(Subpel<T, W> &sp, MV2 t, MV2 diag) {
  if (t.row == sp.best.row && t.col == sp.best.col) return;
  if (t.row == sp.best.row) diag.row *= -1;
  else if (t.col == sp.best.col) diag.col *= -1;
  const MV2 rb = { sp.best.row + diag.row, sp.best.col };
  const MV2 cb = { sp.best.row, sp.best.col + diag.col };
  const MV2 db = { sp.best.row + diag.row, sp.best.col + diag.col };
  int has_better = 0;
  check_better(sp, rb.row, rb.col, true, &has_better);
  check_better(sp, cb.row, cb.col, true, &has_better);
  if (has_better) check_better(sp, db.row, db.col, true, &has_better);
}

// av1_find_best_sub_pixel_tree{,_pruned,_pruned_more} (mcomp.c:2844-3133) with
// cost_list == NULL, forced_stop = EIGHTH_PEL, MV_COST_NONE, unscaled refs.
template <typename T, int W>
__device__ __forceinline__ unsigned subpel_search(Search<T> &S, const KParams &P, MV2 start_full, MV2 *best, T *tmp) {
  Subpel<T, W> sp;
  sp.S = &S;
  sp.bd = P.is_hbd ? P.bit_depth : 8;
  sp.tmp = tmp;
  const int max_mv = 1023 * 8;  // av1_set_subpel_mv_search_range mcomp.h:344-361
  sp.lim.col_min = imax(-(1 << 14) + 1, imax(S.lim.col_min * 8, -max_mv));
  sp.lim.col_max = imin((1 << 14) - 1, imin(S.lim.col_max * 8, max_mv));
  sp.lim.row_min = imax(-(1 << 14) + 1, imax(S.lim.row_min * 8, -max_mv));
  sp.lim.row_max = imin((1 << 14) - 1, imin(S.lim.row_max * 8, max_mv));
  MV2 start = { start_full.row * 8, start_full.col * 8 };
  sp.best = start;
  int hstep = 4;
  if (P.subpel_method == 0) {  // SUBPEL_TREE
    sp.besterr = upsampled_err<T, W>(S, start.row, start.col, sp.bd, tmp);
    const int rounds = P.allow_hp ? 3 : 2;
    for (int iter = 0; iter < rounds; ++iter) {
      const MV2 center = sp.best;
      const MV2 diag = first_level(sp, center, hstep, true);
      if (!(center.row == sp.best.row && center.col == sp.best.col) && P.iters_per_step > 1)
        second_level_v2(sp, center, diag);
      hstep >>= 1;
    }
  } else {
    // every candidate of the stage lies within two full-pel steps of its start: one window for all of them
    if (!window_covers(S, start_full.row, start_full.col, 2))
      window_load<T, W>(S, reinterpret_cast<unsigned char *>(tmp), start_full.row, start_full.col);
    // setup_center_error (mcomp.c:2718-2777): vf(ref, src); the variance is symmetric in its arguments
    sp.besterr = subpel_err_win<T, W>(S, start.row, start.col, 2);
    const int rounds = P.allow_hp ? 3 : 2;
    for (int it = 0; it < rounds; it++) {
      const MV2 center = sp.best;
      const MV2 diag = first_level(sp, center, hstep, false);
      if (P.iters_per_step > 1) second_level_fast(sp, center, diag, hstep);
      hstep >>= 1;
    }
  }
  *best = sp.best;
  return sp.besterr;
}

__device__ __forceinline__ int rawpel(int x) { return (x + 3 + (x >= 0)) >> 3; }  // GET_MV_RAWPEL mv.h:28

// tf_motion_search (temporal_filter.c:87-253) is split along its own data
// dependencies into three kernels (see tf_search32_kernel below):
//   * the ref_mv chain runs through the 32x32 search only (:182-188,:249-252);
//   * the four 16x16 searches of a (block, frame) start from the 32x32 result
//     and are independent of everything else (:190-237);
//   * the partition decision (:245, :270-292) needs both and happens in the
//     filter kernel.
template <typename T>
__device__ __forceinline__ void search_init(Search<T> &S, const KParams &P, int mb_row, int mb_col) {
  S.stride = P.pitch[0];
  S.sad_lambda = P.sad_lambda;
  S.sse_lambda = P.sse_lambda;
  S.hbd_shift = P.hbd_shift;
  S.is_hbd = P.is_hbd;
  S.win = nullptr;
  S.srcs = 0;
  S.wr = S.wc = S.wR = S.wpitch = S.wshift = 0;
  S.ctr = P.ctr;
  S.rs = nullptr;
  // av1_set_mv_{row,col}_limits (mcomp.h:216-240) + av1_set_mv_search_range (mcomp.c:196-215)
  const int border = P.border, mi_row = mb_row * 8, mi_col = mb_col * 8;
  S.lim.row_min = imax(-(mi_row * 4 + border - 8), -(((mi_row + 8) * 4) + 8));
  S.lim.row_max = imin((P.mi_rows - mi_row - 8) * 4 + border - 8, (P.mi_rows - mi_row) * 4 + 8);
  S.lim.col_min = imax(-(mi_col * 4 + border - 8), -(((mi_col + 8) * 4) + 8));
  S.lim.col_max = imin((P.mi_cols - mi_col - 8) * 4 + border - 8, (P.mi_cols - mi_col) * 4 + 8);
  S.lim.col_min = imax(S.lim.col_min, -1023);
  S.lim.col_max = imin(S.lim.col_max, 1023);
  S.lim.row_min = imax(S.lim.row_min, -1023);
  S.lim.row_max = imin(S.lim.row_max, 1023);
}

// Kernel 1: the 32x32 search of every frame of the window, chained through
// ref_mv (temporal_filter.c:855-871).  One warp per 32x32 block.
// Two register budgets of the same code, chosen per launch by the host: MINB = 20 (96 registers,
// 20 warps per SM) when the whole grid is resident at once (<= 148 * 20 blocks, e.g. 1080p), so
// no second partial wave forms; MINB = 12 (168 registers, no spills) for larger grids, where the
// latency-bound chain runs faster per launch and leaves registers for concurrent 16x16 launches.
#ifndef TF_S32_LO
#define TF_S32_LO 12
#endif
#ifndef TF_S32_HI
#define TF_S32_HI 20
#endif
#ifndef TF_S32_HI_HBD
#define TF_S32_HI_HBD 16
#endif
constexpr int S32_WARPS_HI = TF_S32_HI, S32_WARPS_HI_HBD = TF_S32_HI_HBD, S32_WARPS_LO = TF_S32_LO;
#ifndef TF_S16_WARPS
#define TF_S16_WARPS 24
#endif
constexpr int S16_WARPS = TF_S16_WARPS;
template <typename T, int MINB>
__device__ __forceinline__ void search32_block(const KParams &P, const unsigned bid) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int lane = lane_id();
  const int mb_row = P.row_begin + bid / P.mb_cols;
  const int mb_col = bid % P.mb_cols;
  const int blk = mb_row * P.mb_cols + mb_col;
  const int st = P.pitch[0];
  const int y_offset = mb_row * 32 * st + mb_col * 32;
  const T *cur = reinterpret_cast<const T *>(P.frm[P.filter_idx][0]);
  Search<T> S;
  search_init(S, P, mb_row, mb_col);
  S.src = cur + y_offset;
  src_tile_load<T, 32>(S, smem_raw + SearchSmem<T, 32>::WIN);  // once per block: the same source for every frame
  // ref_mv chain (temporal_filter.c:855-871): carried in global memory across launches
  MV2 ref_mv = { 0, 0 };
  if (P.frame_begin > 0) {
    ref_mv.row = P.s_ref_mv[blk * 2 + 0];
    ref_mv.col = P.s_ref_mv[blk * 2 + 1];
  }
  for (int frame = P.frame_begin; frame < P.frame_end; frame++) {
    if (frame == P.filter_idx) {
      ref_mv.row = -ref_mv.row;
      ref_mv.col = -ref_mv.col;
      continue;
    }
    S.ref = reinterpret_cast<const T *>(P.frm[frame][0]) + y_offset;
    const MV2 start = { rawpel(ref_mv.row), rawpel(ref_mv.col) };
    MV2 best_full;
    full_pixel_search<T, 32>(S, P, start, &best_full, smem_raw);
    int block_mse;
    MV2 block_mv;
    if (P.force_integer_mv == 1) {
      unsigned sse;
      const unsigned err =
          variance<T, 32>(S.ref + best_full.row * st + best_full.col, st, S.src, st, S.hbd_shift, &sse);
      block_mse = (int)((err + 512u) / 1024u);
      block_mv.row = best_full.row * 8;
      block_mv.col = best_full.col * 8;
    } else {
      const unsigned err = subpel_search<T, 32>(S, P, best_full, &block_mv, reinterpret_cast<T *>(smem_raw));
      block_mse = (int)((err + 512u) / 1024u);
      ref_mv = block_mv;
    }
    if (lane == 0) {
      const size_t bf = (size_t)blk * P.num_frames + frame;
      P.s_blk_mv[bf * 2 + 0] = (int16_t)block_mv.row;
      P.s_blk_mv[bf * 2 + 1] = (int16_t)block_mv.col;
      P.s_blk_mse[bf] = block_mse;
    }
    if (block_mse > P.mse_thresh) {  // :249-252
      ref_mv.row = 0;
      ref_mv.col = 0;
    }
  }
  if (lane == 0) {
    P.s_ref_mv[blk * 2 + 0] = (int16_t)ref_mv.row;
    P.s_ref_mv[blk * 2 + 1] = (int16_t)ref_mv.col;
  }
}
template <typename T, int MINB>
__global__ void __launch_bounds__(32, MINB) tf_search32_kernel(const __grid_constant__ KParams P) {
  search32_block<T, MINB>(P, blockIdx.x);
}

// Kernel 2: every 16x16 sub-block search is an independent task
// (frame, block, sub-block); it starts from the full-pel rounding of the
// 32x32 result (temporal_filter.c:194) and reuses the 32x32 block's MV limits
// (:202-205).  One warp per task, frame-major task order for L2 locality.
template <typename T>
__device__ __forceinline__ void search16_task(const KParams &P, const int task) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int lane = lane_id();
  const int nblk = (P.row_end - P.row_begin) * P.mb_cols;
  const int fidx = task / (nblk * 4);
  const int rem = task - fidx * nblk * 4;
  const int bl = rem >> 2, sub = rem & 3;
  // frames [frame_begin, frame_end) minus the centre frame, in order
  int frame = P.frame_begin + fidx;
  if (P.filter_idx >= P.frame_begin && frame >= P.filter_idx) frame++;
  const int mb_row = P.row_begin + bl / P.mb_cols;
  const int mb_col = bl % P.mb_cols;
  const int blk = mb_row * P.mb_cols + mb_col;
  const int st = P.pitch[0];
  const int off = mb_row * 32 * st + mb_col * 32 + (sub >> 1) * 16 * st + (sub & 1) * 16;
  Search<T> S;
  search_init(S, P, mb_row, mb_col);
  S.src = reinterpret_cast<const T *>(P.frm[P.filter_idx][0]) + off;
  S.ref = reinterpret_cast<const T *>(P.frm[frame][0]) + off;
  S.rs = P.rs[frame] + off;
  src_tile_load<T, 16>(S, smem_raw + SearchSmem<T, 16>::WIN);
  const size_t bf = (size_t)blk * P.num_frames + frame;
  const MV2 start = { rawpel((int)P.s_blk_mv[bf * 2 + 0]), rawpel((int)P.s_blk_mv[bf * 2 + 1]) };
  MV2 best_full, best;
  full_pixel_search<T, 16>(S, P, start, &best_full, smem_raw);
  const unsigned err = subpel_search<T, 16>(S, P, best_full, &best, reinterpret_cast<T *>(smem_raw));
  if (lane == 0) {
    P.s_sub_mv[(bf * 4 + sub) * 2 + 0] = (int16_t)best.row;
    P.s_sub_mv[(bf * 4 + sub) * 2 + 1] = (int16_t)best.col;
    P.s_sub_mse[bf * 4 + sub] = (int)((err + 128u) / 256u);
  }
}
template <typename T>
__global__ void __launch_bounds__(32, S16_WARPS) tf_search16_kernel(const __grid_constant__ KParams P) {
  search16_task<T>(P, blockIdx.x);
}

// Position rule of a batched search item (tf_gpu.h): the block starts inside the mi grid (it may stick out of it
// like the last 32x32 row of a 1080p frame); x is a multiple of 16 because the SAD engine reads source rows with
// 16-byte loads.  The host checks it for the synchronous calls, tf_motion_batch_kernel for device-memory items.
__host__ __device__ __forceinline__ bool item_position_ok(int x, int y, int mi_rows, int mi_cols) {
  return x >= 0 && y >= 0 && !(x & 15) && !(y & 3) && x < mi_cols * 4 && y < mi_rows * 4;
}

// Batched full-pixel search (tf_gpu_fullpel_search_batch): one warp per item, the engine of the two
// kernels above on an arbitrary block of an arbitrary frame pair.
struct SearchItem {
  int x, y;
  int16_t start_row, start_col;
};
struct SearchResult {
  int16_t row, col;
  int32_t var;
};
// The per-item part of the batched searches: MV limits for a W x W block at mi position (y / 4, x / 4),
// av1_set_mv_{row,col}_limits (mcomp.h:216-240), then av1_set_mv_search_range (mcomp.c:196-215) around a zero
// reference MV; then av1_full_pixel_search from `start` with `ref` as the reference.
// Leaves S set up for the item (source, reference, limits, search window) for what follows.
template <typename T, int W>
__device__ __forceinline__ void item_full_pixel_search(Search<T> &S, const KParams &P, const T *src, const T *ref,
                                                       int x, int y, MV2 start, MV2 *best, unsigned char *smem_raw) {
  search_init(S, P, 0, 0);
  const int border = P.border, mi_row = y >> 2, mi_col = x >> 2, mih = W / 4;
  S.lim.row_min = imax(-(mi_row * 4 + border - 8), -(((mi_row + mih) * 4) + 8));
  S.lim.row_max = imin((P.mi_rows - mi_row - mih) * 4 + border - 8, (P.mi_rows - mi_row) * 4 + 8);
  S.lim.col_min = imax(-(mi_col * 4 + border - 8), -(((mi_col + mih) * 4) + 8));
  S.lim.col_max = imin((P.mi_cols - mi_col - mih) * 4 + border - 8, (P.mi_cols - mi_col) * 4 + 8);
  S.lim.col_min = imax(S.lim.col_min, -1023);
  S.lim.col_max = imin(S.lim.col_max, 1023);
  S.lim.row_min = imax(S.lim.row_min, -1023);
  S.lim.row_max = imin(S.lim.row_max, 1023);
  const int off = y * P.pitch[0] + x;
  S.src = src + off;
  S.ref = ref + off;
  full_pixel_search<T, W>(S, P, start, best, smem_raw);
}
template <typename T, int W>
__global__ void __launch_bounds__(32, W == 32 ? S32_WARPS_LO : 24)
    tf_fullpel_batch_kernel(const __grid_constant__ KParams P, const T *src, const T *ref, const SearchItem *items,
                            SearchResult *results, int n) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int lane = lane_id();
  if ((int)blockIdx.x >= n) return;
  const SearchItem it = items[blockIdx.x];
  Search<T> S;
  const MV2 start = { (int)it.start_row, (int)it.start_col };
  MV2 best;
  item_full_pixel_search<T, W>(S, P, src, ref, it.x, it.y, start, &best, smem_raw);
  const int var = var_cost<T, W>(S, best.row, best.col);
  if (lane == 0) {
    results[blockIdx.x].row = (int16_t)best.row;
    results[blockIdx.x].col = (int16_t)best.col;
    results[blockIdx.x].var = var;
  }
}

// Batched motion search (tf_gpu_motion_search_batch): what tf_motion_search() (temporal_filter.c:145-188) does to
// one block, one warp per item.  Frame 0 of P is the source, frame 1 + item.ref the item's reference.  After the
// full-pel stage of tf_fullpel_batch_kernel the source block is staged as a shared-memory tile (the sub-pel error
// routines read it from there, as in search16_task) and find_fractional_mv_step refines the MV to 1/8 pel in the
// shared memory of the search (MV_COST_NONE, forced_stop = EIGHTH_PEL, no cost list); under force_integer_mv the
// result is the variance at the full-pel MV instead (:162-172).
// Every item is checked before any frame is read (items in device memory are never seen by the host): an item whose
// position fails item_position_ok or whose ref is outside [0, P.num_frames - 1) gets fullpel_var =
// MOTION_REJECTED, MVs 0 and err = UINT32_MAX.
struct MotionItem {
  int x, y;
  int16_t start_row, start_col;
  int32_t ref;
};
struct MotionResult {
  int16_t fullpel_row, fullpel_col;
  int32_t fullpel_var;
  int16_t row, col;
  uint32_t err;
};
constexpr int MOTION_REJECTED = -1;  // TF_GPU_MOTION_REJECTED; a searched item's fullpel_var is never negative
template <typename T, int W>
__global__ void __launch_bounds__(32, W == 32 ? S32_WARPS_LO : 24)
    tf_motion_batch_kernel(const __grid_constant__ KParams P, const MotionItem *items, MotionResult *results, int n) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int lane = lane_id();
  if ((int)blockIdx.x >= n) return;
  const MotionItem it = items[blockIdx.x];
  if (!item_position_ok(it.x, it.y, P.mi_rows, P.mi_cols) || it.ref < 0 || it.ref >= P.num_frames - 1) {
    if (lane == 0) {
      MotionResult r;
      r.fullpel_row = r.fullpel_col = r.row = r.col = 0;
      r.fullpel_var = MOTION_REJECTED;
      r.err = 0xffffffffu;
      results[blockIdx.x] = r;
    }
    return;
  }
  const int f = 1 + it.ref;
  Search<T> S;
  const MV2 start = { (int)it.start_row, (int)it.start_col };
  MV2 best_full;
  item_full_pixel_search<T, W>(S, P, reinterpret_cast<const T *>(P.frm[0][0]), reinterpret_cast<const T *>(P.frm[f][0]),
                               it.x, it.y, start, &best_full, smem_raw);
  const int var = var_cost<T, W>(S, best_full.row, best_full.col);
  src_tile_load<T, W>(S, smem_raw + SearchSmem<T, W>::WIN);
  MV2 mv;
  unsigned err;
  if (P.force_integer_mv == 1) {
    unsigned sse;
    err = variance<T, W>(S.ref + best_full.row * S.stride + best_full.col, S.stride, S.src, S.stride, S.hbd_shift, &sse);
    mv.row = best_full.row * 8;
    mv.col = best_full.col * 8;
  } else {
    err = subpel_search<T, W>(S, P, best_full, &mv, reinterpret_cast<T *>(smem_raw));
  }
  if (lane == 0) {
    MotionResult r;
    r.fullpel_row = (int16_t)best_full.row;
    r.fullpel_col = (int16_t)best_full.col;
    r.fullpel_var = var;
    r.row = (int16_t)mv.row;
    r.col = (int16_t)mv.col;
    r.err = err;
    results[blockIdx.x] = r;
  }
}

// ---------------------------------------------------------------------------
// Predictor: tf_build_predictor (temporal_filter.c:328-390) ->
// init_subpel_params (reconinter.h:131-165) -> convolve_2d_facade_single
// (convolve.c:495-515) with the 12-tap MULTITAP_SHARP2 kernels.
// ---------------------------------------------------------------------------
template <typename T>
__device__ __noinline__ void convolve12(const KParams &P, const T *src, int ss, T *dst, int ds, int w, int h, int sx, int sy,
                           int16_t *im) {
  const int lane = lane_id();
  const int pbd = P.is_hbd ? P.bit_depth : 8;
  int r0b = 3, r1b = 11;  // get_conv_params_no_round (convolve.h:63-95)
  if (P.is_hbd && P.bit_depth + 7 - r0b + 2 > 16) {
    const int d = P.bit_depth + 7 - r0b + 2 - 16;
    r0b += d;
    r1b -= d;
  }
  const int rp = 32 / w;  // rows per iteration (w is 8 or 16)
  const int col = lane % w, rr = lane / w;
  if (!sx && !sy) {  // aom_convolve_copy; h / rp is 4 or 8: all loads in flight
    T v[8];
#pragma unroll
    for (int k = 0; k < 8; k++)
      if (rr + k * rp < h) v[k] = __ldg(src + (rr + k * rp) * ss + col);
#pragma unroll
    for (int k = 0; k < 8; k++)
      if (rr + k * rp < h) dst[(rr + k * rp) * ds + col] = v[k];
  } else if (sx && !sy) {
    const int16_t *f = c_k12[sx];
    const int bits = 7 - r0b;
    for (int y = rr; y < h; y += rp) {
      int res = 0;
#pragma unroll
      for (int k = 0; k < 12; k++) res += f[k] * (int)__ldg(src + y * ss + col - 5 + k);
      res = rpot(res, r0b);
      dst[y * ds + col] = (T)clip_px(rpot(res, bits), pbd);
    }
  } else if (!sx && sy) {
    const int16_t *f = c_k12[sy];
    for (int y = rr; y < h; y += rp) {
      int res = 0;
#pragma unroll
      for (int k = 0; k < 12; k++) res += f[k] * (int)__ldg(src + (y - 5 + k) * ss + col);
      dst[y * ds + col] = (T)clip_px(rpot(res, 7), pbd);
    }
  } else {
    const int16_t *fx = c_k12[sx], *fy = c_k12[sy];
    const int bits = 14 - r0b - r1b;
    for (int y = rr; y < h + 11; y += rp) {
      int sum = 1 << (pbd + 6);
#pragma unroll
      for (int k = 0; k < 12; k++) sum += fx[k] * (int)__ldg(src + (y - 5) * ss + col - 5 + k);
      im[y * w + col] = (int16_t)rpot(sum, r0b);
    }
    __syncwarp();
    const int ob = pbd + 14 - r0b;
    for (int y = rr; y < h; y += rp) {
      int sum = 1 << ob;
#pragma unroll
      for (int k = 0; k < 12; k++) sum += fy[k] * (int)im[(y + k) * w + col];
      int res = rpot(sum, r1b) - ((1 << (ob - r1b)) + (1 << (ob - r1b - 1)));
      if (sizeof(T) == 1) res = (int)(int16_t)res;  // convolve.c:120
      dst[y * ds + col] = (T)clip_px(rpot(res, bits), pbd);
    }
    __syncwarp();
  }
}

// The same three variants for 16-bit containers with two samples per register.  The 12 taps of
// MULTITAP_SHARP2 at a fractional position fit a signed byte (-26 .. 127; 128 only occurs at position 0,
// which is the copy path), the samples (<= 4095) fit a signed halfword, and the 2-D intermediate is narrowed
// to one as the reference's int16_t im_block is (convolve.c:96; at 10 and 12 bit full-range content takes it
// past 32767 and it wraps, here as there), so one IDP.2A does two taps:
//   horizontal stage: a lane produces two adjacent outputs of a row from eight aligned words (the byte
//     parity of the row start is uniform over the warp: one funnel shift per word pair), 12 IDP.2A;
//   the intermediate is stored TRANSPOSED (im[col][row], column pitch h + 12), so the vertical stage reads
//     vertically adjacent values as words: a lane produces two vertically adjacent outputs from seven
//     shared-memory words, 12 IDP.2A;
//   vertical-only positions copy the rows transposed and use the same vertical stage.
// Rounding and offsets are those of convolve12 above, term for term.
__device__ __forceinline__ unsigned pack_taps(const int16_t *f, int k) {
  return ((unsigned)f[k] & 0xffu) | (((unsigned)f[k + 1] & 0xffu) << 8);
}
__device__ __noinline__ void convolve12_packed(const KParams &P, const uint16_t *src, int ss, uint16_t *dst, int ds, int w,
                                               int h, int sx, int sy, int16_t *im) {
  const int lane = lane_id();
  const int pbd = P.bit_depth;
  int r0b = 3, r1b = 11;  // get_conv_params_no_round (convolve.h:63-95)
  if (P.bit_depth + 7 - r0b + 2 > 16) {
    const int d = P.bit_depth + 7 - r0b + 2 - 16;
    r0b += d;
    r1b -= d;
  }
  const int PT = h + 12;  // column pitch of the transposed intermediate (even: columns start word-aligned)
  {
    // stage A
    const int ppr = w >> 1, rpi = 32 / ppr;  // column pairs per row, rows per iteration
    const int pc = lane % ppr, ry = lane / ppr;
    const int nrows = sy ? h + 11 : h;
    const uint16_t *base = src - (sy ? 5 * ss : 0);
    if (sx) {
      unsigned tx[6];
#pragma unroll
      for (int k = 0; k < 6; k++) tx[k] = pack_taps(c_k12[sx], 2 * k);
      const uintptr_t a0 = reinterpret_cast<uintptr_t>(base + 2 * pc - 5);
      const unsigned sh = (a0 & 2) ? 16u : 0u;  // uniform: the pitch and 2 * pc are even
      const unsigned char *row0 = reinterpret_cast<const unsigned char *>(a0 & ~(uintptr_t)3);
      const int off = 1 << (pbd + 6), bits = 7 - r0b;
#pragma unroll 1  // (two or three rows in flight: measured, no change)
      for (int y = ry; y < nrows; y += rpi) {
        const uint32_t *wp = reinterpret_cast<const uint32_t *>(row0 + (size_t)y * ss * 2);
        uint32_t wv[8];
#pragma unroll
        for (int k = 0; k < 8; k++) wv[k] = __ldg(wp + k);
        unsigned pr[7];
#pragma unroll
        for (int k = 0; k < 7; k++) pr[k] = __funnelshift_r(wv[k], wv[k + 1], sh);
        int s0 = 0, s1 = 0;
#pragma unroll
        for (int k = 0; k < 6; k++) {
          s0 = __dp2a_lo((int)pr[k], (int)tx[k], s0);
          s1 = __dp2a_lo((int)__funnelshift_r(pr[k], pr[k + 1], 16), (int)tx[k], s1);
        }
        if (sy) {
          im[(2 * pc) * PT + y] = (int16_t)rpot(s0 + off, r0b);
          im[(2 * pc + 1) * PT + y] = (int16_t)rpot(s1 + off, r0b);
        } else {
          dst[y * ds + 2 * pc] = (uint16_t)clip_px(rpot(rpot(s0, r0b), bits), pbd);
          dst[y * ds + 2 * pc + 1] = (uint16_t)clip_px(rpot(rpot(s1, r0b), bits), pbd);
        }
      }
    } else {  // vertical only: the source rows, transposed
#pragma unroll 1
      for (int y = ry; y < nrows; y += rpi) {
        im[(2 * pc) * PT + y] = (int16_t)__ldg(base + y * ss + 2 * pc);
        im[(2 * pc + 1) * PT + y] = (int16_t)__ldg(base + y * ss + 2 * pc + 1);
      }
    }
  }
  __syncwarp();
  if (!sy) return;
  {
    // stage B
    unsigned ty[6];
#pragma unroll
    for (int k = 0; k < 6; k++) ty[k] = pack_taps(c_k12[sy], 2 * k);
    const int col = lane % w, ypl = lane / w, ypi = 32 / w;
    const int ob = pbd + 14 - r0b, bits = 14 - r0b - r1b;
    const int sub = (1 << (ob - r1b)) + (1 << (ob - r1b - 1));
#pragma unroll 1
    for (int yp = ypl; yp < (h >> 1); yp += ypi) {
      const uint32_t *cp = reinterpret_cast<const uint32_t *>(im + col * PT) + yp;
      uint32_t pv[7];
#pragma unroll
      for (int k = 0; k < 7; k++) pv[k] = cp[k];
      int s0 = 0, s1 = 0;
#pragma unroll
      for (int k = 0; k < 6; k++) {
        s0 = __dp2a_lo((int)pv[k], (int)ty[k], s0);
        s1 = __dp2a_lo((int)__funnelshift_r(pv[k], pv[k + 1], 16), (int)ty[k], s1);
      }
      int v0, v1;
      if (sx) {
        v0 = rpot(rpot(s0 + (1 << ob), r1b) - sub, bits);
        v1 = rpot(rpot(s1 + (1 << ob), r1b) - sub, bits);
      } else {
        v0 = rpot(s0, 7);
        v1 = rpot(s1, 7);
      }
      dst[(2 * yp) * ds + col] = (uint16_t)clip_px(v0, pbd);
      dst[(2 * yp + 1) * ds + col] = (uint16_t)clip_px(v1, pbd);
    }
  }
  __syncwarp();
}

// The filter kernel runs FILT_WARPS = 4 warps per 32x32 block: warp q builds the predictor of
// sub-block q of every plane (its own MV), the element-wise stages stride over all threads.
// seven blocks per SM (73 registers, 48 bytes of spills): filter 2.70 -> 2.64 ms at 4K 10-bit, 0.57 -> 0.51 ms at 1080p 8-bit
#ifndef TF_FILT_MINB
#define TF_FILT_MINB 7
#endif
constexpr int FILT_WARPS = 4;
constexpr int FILT_THREADS = FILT_WARPS * 32;

// The scaled source position of one predictor sub-block: init_subpel_params (reconinter.h:131-165) as
// tf_build_predictor (temporal_filter.c:356-365) calls it for the sub-block at plane position (y, x), with the
// reference's clamp to [-((288 >> ss) - 4), aligned + 4] samples.  Integer sample: pos >> 10; 1/16 phase:
// (pos & 1023) >> 6.
__device__ __forceinline__ void predictor_position(const KParams &P, int k, int y, int x, MV2 mv, int ssy, int ssx,
                                                   int *py, int *px) {
  int pos_y = ((y << 4) + mv.row * (1 << (1 - ssy))) * 64 + 32;
  int pos_x = ((x << 4) + mv.col * (1 << (1 - ssx))) * 64 + 32;
  const int top = -(((288 >> ssy) - 4) << 10), left = -(((288 >> ssx) - 4) << 10);
  *py = iclamp(pos_y, top, (P.aligned_h[k] + 4) << 10);
  *px = iclamp(pos_x, left, (P.aligned_w[k] + 4) << 10);
}

template <typename T>
__device__ void build_predictor(const KParams &P, const T *const ref[3], int mb_row, int mb_col, const MV2 *mvs,
                                T *pred, int16_t *im /* this warp's scratch */) {
  const int q = threadIdx.x >> 5;  // sub-block of this warp, raster order (temporal_filter.c:366-385)
  const MV2 mv = mvs[q];
  int plane_offset = 0;
  for (int plane = 0; plane < P.num_planes; plane++) {
    const int ssy = plane ? P.ss_y : 0, ssx = plane ? P.ss_x : 0;
    const int k = plane > 0;
    const int plane_h = 32 >> ssy, plane_w = 32 >> ssx;
    const int plane_y = (32 * mb_row) >> ssy, plane_x = (32 * mb_col) >> ssx;
    const int h = plane_h >> 1, w = plane_w >> 1;
    const int i = (q >> 1) * h, j = (q & 1) * w;
    int pos_y, pos_x;
    predictor_position(P, k, plane_y + i, plane_x + j, mv, ssy, ssx, &pos_y, &pos_x);
    const T *src = ref[plane] + (pos_y >> 10) * P.pitch[k] + (pos_x >> 10);
    const int sxp = (pos_x & 1023) >> 6, syp = (pos_y & 1023) >> 6;
    if constexpr (sizeof(T) == 2) {
      if (sxp | syp) convolve12_packed(P, src, P.pitch[k], &pred[plane_offset + i * plane_w + j], plane_w, w, h, sxp, syp, im);
      else convolve12<T>(P, src, P.pitch[k], &pred[plane_offset + i * plane_w + j], plane_w, w, h, 0, 0, im);
    } else {
      convolve12<T>(P, src, P.pitch[k], &pred[plane_offset + i * plane_w + j], plane_w, w, h, sxp, syp, im);
    }
    plane_offset += plane_h * plane_w;
  }
  __syncthreads();
}

// ---------------------------------------------------------------------------
// Weights: av1_apply_temporal_filter_c (temporal_filter.c:557-707)
// sq:   block-shared u32[1024] (horizontal 5-sums of the squared differences of the current plane)
// lsum: block-shared u32[1024] (raw luma squared differences, read by the chroma planes)
//
// Every thread owns the same pixels in every stage: pixel idx = tid + k * NT of a plane, i.e. column
// j = tid % w and rows r0 + k * (NT / w).  The lanes of a row are adjacent lanes of one warp (w = 32:
// the warp, w = 16: a half warp), so the horizontal 5-sum with edge clamp (:463-493 window, clamped as
// the reference clamps the coordinates) is four shuffles, the vertical one five conflict-free shared
// loads of a column; the chroma planes add the co-located luma squares from lsum.
//
// The weight (int)(exp(-scaled_error) * 1000) (:691-693) is computed in fp64 with the reference's
// operation order.  (An fp32 ex2.approx fast path with an exact fp64 fallback near integer boundaries was
// measured: 10 % fewer instructions in this kernel, no gain in time -- the kernel is bound by shared-memory
// / L1 wavefronts and latency, not by the fp64 pipe -- so the single exact path stays.)
// ---------------------------------------------------------------------------
__device__ __forceinline__ int tf_weight(double scaled_error) {
  return (int)__dmul_rn(exp(-scaled_error), 1000.0);
}

template <typename T>
__device__ void apply_filter(const KParams &P, const T *curb, int mb_row, int mb_col, const MV2 *mvs,
                             const int *mses, const T *pred, uint32_t *accum, uint16_t *count, uint32_t *sq,
                             uint32_t *lsum, const double *terms /* shared: d_factor[4], block_error * inv_factor [4] */) {
  constexpr int NT = FILT_THREADS;
  constexpr int MAXPX = 1024 / NT;  // pixels of one plane per thread
  const int tid = threadIdx.x, lane = tid & 31;
  const double inv_factor = 1.0 / ((5 + 1) * 20);
  const double weight_factor = (double)5 * inv_factor;
  (void)mvs;
  (void)mses;
  (void)inv_factor;
  (void)mb_row;
  (void)mb_col;
  int plane_offset = 0;
  for (int plane = 0; plane < P.num_planes; plane++) {
    const int ssy = plane ? P.ss_y : 0, ssx = plane ? P.ss_x : 0;
    const int h = 32 >> ssy, w = 32 >> ssx, n = h * w, wsh = 5 - ssx;
    const int rpp = NT >> wsh;    // rows per pass over the plane
    const int npass = n / NT;     // 8 (32x32), 4 (16x32), 2 (16x16)
    const int j = tid & (w - 1), r0 = tid >> wsh;
    const int num_ref_pixels = 25 + (plane ? (1 << (ssx + ssy)) : 0);
    const double inv_num_ref_pixels = 1.0 / num_ref_pixels;
    // lanes holding the horizontal neighbours of this pixel's row, edge-clamped
    const int seg = lane & ~(w - 1);
    const int l_m2 = seg + imax(j - 2, 0), l_m1 = seg + imax(j - 1, 0);
    const int l_p1 = seg + imin(j + 1, w - 1), l_p2 = seg + imin(j + 2, w - 1);
    // compute_square_diff (:463-493) + horizontal 5-sums
#pragma unroll
    for (int k = 0; k < MAXPX; k++) {
      if (k < npass) {
        const int idx = tid + k * NT;  // == (r0 + k * rpp) * w + j
        const int d = (int)curb[plane_offset + idx] - (int)pred[plane_offset + idx];
        const uint32_t v = (uint32_t)(d * d);
        if (plane == 0 && P.num_planes > 1) lsum[idx] = v;
        const uint32_t h5 = v + __shfl_sync(FULL, v, l_m2) + __shfl_sync(FULL, v, l_m1) + __shfl_sync(FULL, v, l_p1) +
                            __shfl_sync(FULL, v, l_p2);
        sq[idx] = h5;
      }
    }
    __syncthreads();
    const int hbd_sh = P.bit_depth > 8 ? (P.bit_depth - 8) * 2 : 0;
    const int sb_col = (j >= w / 2);
    // a thread's pixels lie in one column half, i.e. in two sub-blocks: the upper and the lower one
    const double d_factor[2] = { terms[sb_col], terms[2 + sb_col] };
    const double b_term[2] = { terms[4 + sb_col], terms[6 + sb_col] };
    // Not unrolled: the filter kernel shrinks from 64 to 40 KB of code (its instruction-cache request rate was 89% of
    // peak) and loses its spills: 2.85 -> 2.65 ms at 4K 10-bit.
#pragma unroll 1
    for (int k = 0; k < MAXPX; k++) {
      if (k < npass) {
        const int i = r0 + k * rpp, idx = tid + k * NT;
        // 25 (+4) squares of at most 4095^2: fits 32 bits
        uint32_t sum_square_diff = sq[imax(i - 2, 0) * w + j] + sq[imax(i - 1, 0) * w + j] + sq[idx] +
                                   sq[imin(i + 1, h - 1) * w + j] + sq[imin(i + 2, h - 1) * w + j];
        if (plane) {  // compute_luma_sq_error_sum (:507-522) on the fly
          for (int ii = 0; ii < (1 << ssy); ii++)
            for (int jj = 0; jj < (1 << ssx); jj++) sum_square_diff += lsum[((i << ssy) + ii) * 32 + (j << ssx) + jj];
        }
        sum_square_diff >>= hbd_sh;
        const double window_error = __dmul_rn((double)sum_square_diff, inv_num_ref_pixels);
        const int sb = (i >= h / 2);  // rows ascend with k: the first half of the passes is the upper sub-block
        const double combined_error = __dadd_rn(__dmul_rn(weight_factor, window_error), b_term[sb]);
        double scaled_error = __dmul_rn(__dmul_rn(combined_error, d_factor[sb]), P.decay[plane]);
        scaled_error = scaled_error < 7.0 ? scaled_error : 7.0;
        const int weight = tf_weight(scaled_error);
        const int pidx = plane_offset + idx;
        accum[pidx] += (uint32_t)(weight * (int)pred[pidx]);
        count[pidx] = (uint16_t)(count[pidx] + weight);
      }
    }
    __syncthreads();
    plane_offset += n;
  }
}

// ---------------------------------------------------------------------------
// Kernel 3: per 32x32 block, for every frame of the window: partition decision,
// predictor, weights, accumulate; then normalise and FRAME_DIFF
// (av1_tf_do_filtering_row, temporal_filter.c:857-937).  accum / count / pred
// never leave shared memory.
// Block-private shared memory, carved at run time (num_pels = 1024 luma + chroma:
// 1536 for 4:2:0, 2048 for 4:2:2, 3072 for 4:4:4):
//   accum u32[num_pels] | sq u32[1024] | lsum u32[1024] | count u16[num_pels] |
//   pred (T view of u16[num_pels]) | cur (T view of u16[num_pels]) | im i16[FILT_WARPS][27*16] | red u64[FILT_WARPS]
// ---------------------------------------------------------------------------
struct WarpSmem {
  double *terms;  // per frame: d_factor of the four sub-blocks, then block_error * inv_factor
  uint32_t *accum, *sq, *lsum;
  uint16_t *count, *pred, *cur;  // cur: the block of the frame to filter, in pred's layout (read once per block)
  int16_t *im;
  unsigned long long *red;
};
constexpr int FILT_IM = (16 + 12) * 16;  // intermediate of one 2-D 12-tap sub-block (transposed form: 16 columns of pitch 28)
__host__ __device__ inline size_t filter_smem_bytes(int num_pels) {
  return (size_t)num_pels * 10 + 2 * 1024 * 4 + FILT_WARPS * FILT_IM * 2 + FILT_WARPS * 8 + 8 * 8;
}
__device__ __forceinline__ WarpSmem carve_smem(unsigned char *raw, int num_pels) {
  WarpSmem sm;
  sm.red = reinterpret_cast<unsigned long long *>(raw);
  sm.terms = reinterpret_cast<double *>(sm.red + FILT_WARPS);
  sm.accum = reinterpret_cast<uint32_t *>(sm.terms + 8);
  sm.sq = sm.accum + num_pels;
  sm.lsum = sm.sq + 1024;
  sm.count = reinterpret_cast<uint16_t *>(sm.lsum + 1024);
  sm.pred = sm.count + num_pels;
  sm.cur = sm.pred + num_pels;
  sm.im = reinterpret_cast<int16_t *>(sm.cur + num_pels);
  return sm;
}

template <typename T>
__device__ __forceinline__ void filter_block(const KParams &P, const unsigned bid) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr int NT = FILT_THREADS;
  const WarpSmem sm = carve_smem(smem_raw, P.num_pels);
  const int tid = threadIdx.x;
  const int mb_row = P.row_begin + bid / P.mb_cols;
  const int mb_col = bid % P.mb_cols;
  const int blk = mb_row * P.mb_cols + mb_col;
  T *pred = reinterpret_cast<T *>(sm.pred);

  for (int i = tid; i < P.num_pels; i += NT) {
    sm.accum[i] = 0;
    sm.count[i] = 0;
  }
  const T *cur[3];
  for (int pl = 0; pl < 3; pl++) cur[pl] = reinterpret_cast<const T *>(P.frm[P.filter_idx][pl]);
  // the block of the frame to filter is compared with the predictor of every frame: one global read
  T *curb = reinterpret_cast<T *>(sm.cur);
  {
    int off = 0;
    for (int pl = 0; pl < P.num_planes; pl++) {
      const int h = 32 >> (pl ? P.ss_y : 0), w = 32 >> (pl ? P.ss_x : 0), st = P.pitch[pl > 0];
      const int wsh = 5 - (pl ? P.ss_x : 0);
      const T *b = cur[pl] + mb_row * h * st + mb_col * w;
      for (int idx = tid; idx < h * w; idx += NT) curb[off + idx] = __ldg(b + (idx >> wsh) * st + (idx & (w - 1)));
      off += h * w;
    }
  }
  __syncthreads();

  for (int frame = 0; frame < P.num_frames; frame++) {
    if (frame == P.filter_idx) {
      // tf_apply_temporal_filter_self (:406-446)
      int off = 0;
      for (int pl = 0; pl < P.num_planes; pl++) {
        const int h = 32 >> (pl ? P.ss_y : 0), w = 32 >> (pl ? P.ss_x : 0), st = P.pitch[pl > 0];
        const int wsh = 5 - (pl ? P.ss_x : 0);
        (void)st;
        (void)wsh;
        for (int idx = tid; idx < h * w; idx += NT) {
          sm.accum[off + idx] += 1000u * (uint32_t)curb[off + idx];
          sm.count[off + idx] = (uint16_t)(sm.count[off + idx] + 1000);
        }
        off += h * w;
      }
      __syncthreads();
      continue;
    }
    const T *ref[3];
    for (int pl = 0; pl < 3; pl++) ref[pl] = reinterpret_cast<const T *>(P.frm[frame][pl]);
    const size_t bf = (size_t)blk * P.num_frames + frame;
    MV2 sub_mvs[4];
    int sub_mses[4];
    const MV2 block_mv = { (int)P.s_blk_mv[bf * 2 + 0], (int)P.s_blk_mv[bf * 2 + 1] };
    const int block_mse = P.s_blk_mse[bf];
#pragma unroll
    for (int i = 0; i < 4; i++) {
      if (P.force_integer_mv == 1) {  // :861-862: the sub-block arrays keep their initial values
        sub_mvs[i].row = sub_mvs[i].col = 0;
        sub_mses[i] = INT_MAX_;
      } else {
        sub_mvs[i].row = (int)P.s_sub_mv[(bf * 4 + i) * 2 + 0];
        sub_mvs[i].col = (int)P.s_sub_mv[(bf * 4 + i) * 2 + 1];
        sub_mses[i] = P.s_sub_mse[bf * 4 + i];
      }
    }
    {  // tf_determine_block_partition (:270-292)
      int mn = INT_MAX_, mx = -INT_MAX_ - 1;
      long long sum = 0;
#pragma unroll
      for (int i = 0; i < 4; i++) {
        sum += sub_mses[i];
        mn = imin(mn, sub_mses[i]);
        mx = imax(mx, sub_mses[i]);
      }
      if ((((long long)block_mse * 15 < sum * 4) && mx - mn < 48) ||
          (((long long)block_mse * 14 < sum * 4) && mx - mn < 24)) {
#pragma unroll
        for (int i = 0; i < 4; i++) {
          sub_mvs[i] = block_mv;
          sub_mses[i] = block_mse;
        }
      }
    }
    if (tid < 4) {  // the distance and block-error terms of the weight (temporal_filter.c:616-625,676-678), once per frame
      const double distance = sqrt((double)(sub_mvs[tid].row * sub_mvs[tid].row + sub_mvs[tid].col * sub_mvs[tid].col));
      const double d = distance / P.dist_thr;
      sm.terms[tid] = d > 1.0 ? d : 1.0;
      sm.terms[4 + tid] = __dmul_rn((double)sub_mses[tid], 1.0 / ((5 + 1) * 20));
    }
    build_predictor<T>(P, ref, mb_row, mb_col, sub_mvs, pred, sm.im + (tid >> 5) * FILT_IM);
    if (P.d_mvs && tid == 0) {
#pragma unroll
      for (int i = 0; i < 4; i++) {
        P.d_mvs[(bf * 4 + i) * 2 + 0] = (int16_t)sub_mvs[i].row;
        P.d_mvs[(bf * 4 + i) * 2 + 1] = (int16_t)sub_mvs[i].col;
      }
    }
    if (P.d_mses && tid == 0) {
#pragma unroll
      for (int i = 0; i < 4; i++) P.d_mses[bf * 4 + i] = sub_mses[i];
    }
    if (P.d_pred)
      for (int i = tid; i < P.num_pels; i += NT) P.d_pred[bf * P.num_pels + i] = (uint16_t)pred[i];
    apply_filter<T>(P, curb, mb_row, mb_col, sub_mvs, sub_mses, pred, sm.accum, sm.count, sm.sq, sm.lsum, sm.terms);
  }

  // tf_normalize_filtered_frame (:740-777); OD_DIVU == integer division here
  // (proved exhaustively against the reference for count in [1000,1023]).
  // FRAME_DIFF (:921-937): vf(src, out, &sse) on the 32x32 luma block, fused into the luma pass.
  unsigned sse = 0;
  {
    int off = 0;
    for (int pl = 0; pl < P.num_planes; pl++) {
      const int h = 32 >> (pl ? P.ss_y : 0), w = 32 >> (pl ? P.ss_x : 0), st = P.out_pitch[pl > 0];
      const int wsh = 5 - (pl ? P.ss_x : 0);
      T *o = reinterpret_cast<T *>(P.out[pl]) + mb_row * h * st + mb_col * w;
      for (int idx = tid; idx < h * w; idx += NT) {
        const int i = idx >> wsh, j = idx & (w - 1);  // w is 32 or 16
        const uint32_t c = sm.count[off + idx];
        const uint32_t v = (sm.accum[off + idx] + (c >> 1)) / c;
        o[i * st + j] = (T)v;
        if (pl == 0 && P.compute_diff) {
          const int d = (int)curb[off + idx] - (int)v;
          sse += (unsigned)(d * d);
        }
      }
      off += h * w;
    }
  }
  if (P.d_accum)
    for (int i = tid; i < P.num_pels; i += NT) P.d_accum[(size_t)blk * P.num_pels + i] = sm.accum[i];
  if (P.d_count)
    for (int i = tid; i < P.num_pels; i += NT) P.d_count[(size_t)blk * P.num_pels + i] = sm.count[i];

  if (P.compute_diff) {
    const unsigned long long w64 = warp_sum_u64((unsigned long long)sse);
    if ((tid & 31) == 0) sm.red[tid >> 5] = w64;
    __syncthreads();
    if (tid == 0) {
      unsigned long long sse64 = 0;
#pragma unroll
      for (int q = 0; q < FILT_WARPS; q++) sse64 += sm.red[q];
      unsigned sse32;
      if (P.hbd_shift == 0) sse32 = (unsigned)sse64;
      else sse32 = (unsigned)((sse64 + ((1ull << (2 * P.hbd_shift)) >> 1)) >> (2 * P.hbd_shift));
      atomicAdd(&P.diff[0], (unsigned long long)sse32);
      atomicAdd(&P.diff[1], (unsigned long long)((long long)sse32 * (long long)sse32));
    }
  }
}
template <typename T>
__global__ void __launch_bounds__(FILT_THREADS, TF_FILT_MINB) tf_filter_kernel(const __grid_constant__ KParams P) {
  filter_block<T>(P, blockIdx.x);
}

// ---------------------------------------------------------------------------
// Predictor at caller MVs (tf_gpu_predict_device): what build_predictor makes of one 16x16 luma unit and its chroma
// sub-blocks, for an item of size 16 or one quadrant of an item of size 32 (each quadrant at the item's MV, from its
// own origin, as the filter predicts a block it did not split).  One warp per unit, FILT_WARPS warps per CTA: an item
// of size 32 is one CTA, warp q its quadrant q; items of size 16 are four to a CTA.  Frame r of P is ref_ids[r].
//
// Far MVs: the reference's clamp lets the origin reach 284 samples (luma) above / left of the frame, past the slot's
// border b.  Each axis of the origin is first clamped to [-b + 5 + PRED_ML, aligned + b - w - 6 - PRED_MR], w the
// sub-block's extent on that axis.  The 12-tap footprint of origin s is [s - 5, s + w + 6); the convolve routines'
// loads reach PRED_ML samples before and PRED_MR after it (convolve12_packed's aligned word loads: a row starts at
// most one sample early, and 8 words from there end at most 3 samples late; convolve12 and the vertical taps read
// the footprint exactly).  When the clamp moves an origin, both footprints lie in the edge-replicated region of that
// axis (x <= 0 or x >= aligned - 1 >= crop - 1) because b >= w + 11 + PRED_ML + PRED_MR, so every sample the
// convolve reads is the one it would read on an unbounded border; every load stays inside the slot, so the __ldg
// loads only ever see the slot's global memory.
// Each sub-block is built in shared memory, as in the filter, and then copied out: the convolve routines get the same
// kinds of pointers from every caller, so adding this caller leaves the filter kernels' code as it was (a direct
// store to `pred` changed their register allocation).
// Rejected items (position rule of item_position_ok, or ref outside [0, num_frames)) get MOTION_REJECTED and zeros.
// ---------------------------------------------------------------------------
constexpr int PRED_ML = 1, PRED_MR = 3;
constexpr int PRED_UNIT_PELS = 16 * 16;  // one sub-block of one plane, staged in shared memory
struct PredictItem {
  int x, y;
  int16_t row, col;
  int32_t ref;
};
template <typename T>
__global__ void __launch_bounds__(FILT_THREADS) tf_predict_kernel(const __grid_constant__ KParams P, const PredictItem *items,
                                                                  T *pred, int32_t *status, int n, int bsize,
                                                                  int border_x_uv, int border_y_uv, int border_luma) {
  __shared__ __align__(16) int16_t im_all[FILT_WARPS * FILT_IM];
  __shared__ __align__(16) T stage_all[FILT_WARPS * PRED_UNIT_PELS];
  const int warp = threadIdx.x >> 5, lane = lane_id();
  const int q = bsize == 32 ? warp : 0;
  const long long item = bsize == 32 ? (long long)blockIdx.x : (long long)blockIdx.x * FILT_WARPS + warp;
  if (item >= n) return;
  const PredictItem it = items[item];
  const bool ok = item_position_ok(it.x, it.y, P.mi_rows, P.mi_cols) && it.ref >= 0 && it.ref < P.num_frames;
  if (q == 0 && lane == 0) status[item] = ok ? 0 : MOTION_REJECTED;
  const MV2 mv = { (int)it.row, (int)it.col };
  T *out = pred + (size_t)item * P.num_pels;
  int16_t *im = im_all + warp * FILT_IM;
  T *stage = stage_all + warp * PRED_UNIT_PELS;
  int plane_offset = 0;
  for (int plane = 0; plane < P.num_planes; plane++) {
    const int ssy = plane ? P.ss_y : 0, ssx = plane ? P.ss_x : 0;
    const int k = plane > 0;
    const int plane_h = bsize >> ssy, plane_w = bsize >> ssx;
    const int h = 16 >> ssy, w = 16 >> ssx;
    const int i = (q >> 1) * h, j = (q & 1) * w;
    if (ok) {
      int pos_y, pos_x;
      predictor_position(P, k, (it.y >> ssy) + i, (it.x >> ssx) + j, mv, ssy, ssx, &pos_y, &pos_x);
      const int by = k ? border_y_uv : border_luma, bx = k ? border_x_uv : border_luma;
      const int oy = iclamp(pos_y >> 10, -by + 5 + PRED_ML, P.aligned_h[k] + by - h - 6 - PRED_MR);
      const int ox = iclamp(pos_x >> 10, -bx + 5 + PRED_ML, P.aligned_w[k] + bx - w - 6 - PRED_MR);
      const T *src = reinterpret_cast<const T *>(P.frm[it.ref][plane]) + oy * P.pitch[k] + ox;
      const int sxp = (pos_x & 1023) >> 6, syp = (pos_y & 1023) >> 6;
      if constexpr (sizeof(T) == 2) {
        if (sxp | syp) convolve12_packed(P, src, P.pitch[k], stage, w, w, h, sxp, syp, im);
        else convolve12<T>(P, src, P.pitch[k], stage, w, w, h, 0, 0, im);
      } else {
        convolve12<T>(P, src, P.pitch[k], stage, w, w, h, sxp, syp, im);
      }
      __syncwarp();
    }
    T *dst = out + plane_offset + i * plane_w + j;
    const int wsh = 4 - ssx;  // w = 1 << wsh
#pragma unroll
    for (int e = lane; e < PRED_UNIT_PELS; e += 32)
      if (e < h * w) dst[(e >> wsh) * plane_w + (e & (w - 1))] = ok ? stage[e] : (T)0;
    __syncwarp();
    plane_offset += plane_h * plane_w;
  }
}

// ---------------------------------------------------------------------------
// Batched windows (tf_gpu_filter_batch_async): several windows over one frame geometry in one grid per kernel,
// blockIdx.y = window.  Each window's KParams carries its own frames, search scratch, output planes and FRAME_DIFF
// slot, so the bodies above run unchanged.  The per-window parameters are the kernel parameter itself
// (__grid_constant__): the window index is warp-uniform, so the window's fields are read with LDCU at a uniform-register
// offset (blockIdx.y * sizeof(KParams)), constant-bank loads like the single-window kernels' immediate-offset ones, no
// extra global traffic.  The host fills only the entries of the windows that have work for the kernel.
// ---------------------------------------------------------------------------
constexpr int MAXB = 16;  // TF_GPU_MAX_BATCH
struct KParamsBatch {
  KParams w[MAXB];
};
static_assert(sizeof(KParamsBatch) <= 32764, "the per-window parameters of a full batch must fit the kernel-parameter limit");

// The 32x32 search of every frame of each window in one launch (the fused chain: the warp walks frames
// [0, num_frames) of its (window, block)).
template <typename T, int MINB>
__global__ void __launch_bounds__(32, MINB) tf_search32_batch_kernel(const __grid_constant__ KParamsBatch B) {
  search32_block<T, MINB>(B.w[blockIdx.y], blockIdx.x);
}
// The 16x16 tasks of every window: grid x covers the window with the most reference frames; the tasks beyond a
// window's own reference frames exit at once.
template <typename T>
__global__ void __launch_bounds__(32, S16_WARPS) tf_search16_batch_kernel(const __grid_constant__ KParamsBatch B) {
  const KParams &P = B.w[blockIdx.y];
  if ((int)blockIdx.x >= (P.row_end - P.row_begin) * P.mb_cols * 4 * (P.num_frames - 1)) return;
  search16_task<T>(P, blockIdx.x);
}
template <typename T>
__global__ void __launch_bounds__(FILT_THREADS, TF_FILT_MINB) tf_filter_batch_kernel(const __grid_constant__ KParamsBatch B) {
  filter_block<T>(B.w[blockIdx.y], blockIdx.x);
}

// ---------------------------------------------------------------------------
// Border replication: av1_copy_and_extend_frame (av1/encoder/extend.c:113-163)
// rebuilt on the device over the device-side border of bx columns / by rows.
// One thread per destination sample outside the crop rectangle.
// ---------------------------------------------------------------------------
template <typename T>
__global__ void extend_borders_kernel(T *plane /* pixel (0,0) */, int pitch, int crop_w, int crop_h, int bx, int by,
                                      int ext_w /* samples right of x=0 incl. crop */, int ext_h) {
  // Only the samples outside the crop rectangle are visited: the side strips of the crop rows
  // first, then the full-width rows above and below.
  const int tw = bx + ext_w;                // total columns covered
  const int sw = bx + (ext_w - crop_w);     // strip samples per crop row (left + right)
  const int n_side = crop_h * sw;
  const int n = n_side + (by + ext_h - crop_h) * tw;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    int x, y;
    if (i < n_side) {
      y = i / sw;
      const int xx = i - y * sw;
      x = xx < bx ? xx - bx : crop_w + (xx - bx);
    } else {
      const int j = i - n_side, ry = j / tw;
      x = j - ry * tw - bx;
      y = ry < by ? ry - by : crop_h + (ry - by);
    }
    const int sx = iclamp(x, 0, crop_w - 1), sy = iclamp(y, 0, crop_h - 1);
    plane[(long long)y * pitch + x] = plane[(long long)sy * pitch + sx];
  }
}

// ---------------------------------------------------------------------------
// Device ingest: a caller's device plane (any row stride, any base alignment)
// copied into a cache slot together with the border replication, in one pass.
// Writes rows [-by, aligned_h + by) x columns [-bx, aligned_w + bx) -- the
// rectangle upload + extend_borders_kernel define -- with
// dst[y][x] = src[clamp(y, 0, crop_h - 1)][clamp(x, 0, crop_w - 1)].
// One thread per 16-byte group of a slot row, counted from the row start
// (column -bx; slot rows are 128-sample aligned), so every store is one
// st.global.v4; the last group of a row may run into the pitch padding,
// which nothing reads.  Loads are as wide as the source address allows
// (16 / 8 / 4 bytes) for groups inside the crop columns, single samples with
// clamping otherwise.  INGEST_ROWS rows per thread for independent loads.
// ---------------------------------------------------------------------------
constexpr int INGEST_THREADS = 128, INGEST_ROWS = 4;

template <typename T>
__global__ void __launch_bounds__(INGEST_THREADS) ingest_plane_kernel(
    T *__restrict__ dst /* slot pixel (0,0) */, int pitch, const T *__restrict__ src /* pixel (0,0) */, int stride,
    int crop_w, int crop_h, int bx, int by, int ext_w /* aligned_w + bx */, int ext_h /* aligned_h + by */) {
  constexpr int V = 16 / sizeof(T);  // samples per group
  constexpr int PER_WORD = 4 / sizeof(T);
  const int groups = (bx + ext_w + V - 1) / V;
  const int g = blockIdx.x * INGEST_THREADS + threadIdx.x;
  if (g >= groups) return;
  const int x0 = g * V - bx;
  const bool inside = x0 >= 0 && x0 + V <= crop_w;
#pragma unroll
  for (int r = 0; r < INGEST_ROWS; r++) {
    const int y = (blockIdx.y * INGEST_ROWS + r) - by;
    if (y >= ext_h) break;
    const T *row = src + (long long)iclamp(y, 0, crop_h - 1) * stride;
    uint32_t w[4];
    const uintptr_t a = (uintptr_t)(row + x0);
    if (inside && (a & 15) == 0) {
      const uint4 q = __ldg((const uint4 *)a);
      w[0] = q.x, w[1] = q.y, w[2] = q.z, w[3] = q.w;
    } else if (inside && (a & 7) == 0) {
      const uint2 q0 = __ldg((const uint2 *)a), q1 = __ldg((const uint2 *)a + 1);
      w[0] = q0.x, w[1] = q0.y, w[2] = q1.x, w[3] = q1.y;
    } else if (inside && (a & 3) == 0) {
#pragma unroll
      for (int j = 0; j < 4; j++) w[j] = __ldg((const uint32_t *)a + j);
    } else {
#pragma unroll
      for (int j = 0; j < 4; j++) {
        uint32_t v = 0;
#pragma unroll
        for (int i = 0; i < PER_WORD; i++)
          v |= (uint32_t)__ldg(row + iclamp(x0 + j * PER_WORD + i, 0, crop_w - 1)) << (8 * sizeof(T) * i);
        w[j] = v;
      }
    }
    *(uint4 *)(dst + (long long)y * pitch + x0) = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

// ---------------------------------------------------------------------------
// Row sums of a cached luma plane for the lower bound of the 16x16 search (diamond_search):
// rs[y][x] = sum of plane[y][x + t], t < 16, for the row blockIdx.y - by and columns [-bx, w - bx).  16 * 4095 fits
// uint16.  One thread per 16 consecutive columns, a running sum along them; with w = aligned_w + 2 bx - 15 every
// stored sum covers columns the upload defines.
// ---------------------------------------------------------------------------
constexpr int ROWSUM_THREADS = 128;

template <typename T>
__global__ void __launch_bounds__(ROWSUM_THREADS) rowsum16_kernel(const T *__restrict__ p00, int pitch,
                                                                  uint16_t *__restrict__ rs00, int bx, int by, int w) {
  const int c0 = (blockIdx.x * ROWSUM_THREADS + threadIdx.x) * 16;  // counted from column -bx
  if (c0 >= w) return;
  const long long at = (long long)((int)blockIdx.y - by) * pitch - bx + c0;
  // samples c0 .. c0 + 31 as 16-byte loads: slot rows start 128-sample aligned at column -bx.  The last group of a
  // row may read up to 16 samples past the defined columns (pitch padding or the next row, inside the allocation:
  // the slot has 2 slack rows); they only reach sums that are not stored.
  constexpr int V = 16 / (int)sizeof(T);
  T x[32];
#pragma unroll
  for (int q = 0; q < 32 / V; q++) *reinterpret_cast<uint4 *>(x + q * V) = __ldg(reinterpret_cast<const uint4 *>(p00 + at) + q);
  unsigned s = 0;
#pragma unroll
  for (int t = 0; t < 16; t++) s += x[t];
  uint32_t o[8];
#pragma unroll
  for (int i = 0; i < 16; i++) {
    if (i > 0) s += (unsigned)x[i + 15] - (unsigned)x[i - 1];
    if (i & 1) o[i >> 1] |= s << 16;
    else o[i >> 1] = s;
  }
  uint16_t *dst = rs00 + at;
  if (w - c0 >= 16) {
    reinterpret_cast<uint4 *>(dst)[0] = make_uint4(o[0], o[1], o[2], o[3]);
    reinterpret_cast<uint4 *>(dst)[1] = make_uint4(o[4], o[5], o[6], o[7]);
  } else {
    for (int i = 0; i < w - c0; i++) dst[i] = (uint16_t)(o[i >> 1] >> (16 * (i & 1)));
  }
}

// ---------------------------------------------------------------------------
// av1_estimate_noise_from_single_plane (temporal_filter.c:1150-1194):
// integer accumulate / count; the final double division is done on the host.
// ---------------------------------------------------------------------------
template <typename T>
__global__ void noise_kernel(const T *src, int pitch, int width, int height, int bd, int edge_thresh,
                             unsigned long long *accum_count /* [2] */) {
  long long acc = 0;
  unsigned cnt = 0;
  const int iw = width - 2, ih = height - 2;
  const long long n = (long long)iw * ih;
  for (long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x; q < n; q += (long long)gridDim.x * blockDim.x) {
    const int i = (int)(q / iw) + 1, j = (int)(q % iw) + 1;
    const T *m = src + (long long)i * pitch + j;
    const int a = m[-pitch - 1], b = m[-pitch], c = m[-pitch + 1];
    const int d = m[-1], e = m[0], f = m[1];
    const int g = m[pitch - 1], h = m[pitch], k = m[pitch + 1];
    const int Gx = (a - c) + (g - k) + 2 * (d - f);
    const int Gy = (a - g) + (c - k) + 2 * (b - h);
    const int Ga = rpot(iabs(Gx) + iabs(Gy), bd - 8);
    if (Ga < edge_thresh) {
      const int v = 4 * e - 2 * (b + h + d + f) + (a + c + g + k);
      acc += rpot(iabs(v), bd - 8);
      ++cnt;
    }
  }
  acc = (long long)warp_sum_u64((unsigned long long)acc);
  cnt = seg_reduce_u32<32>(cnt);
  if ((threadIdx.x & 31) == 0 && cnt) {
    atomicAdd(&accum_count[0], (unsigned long long)acc);
    atomicAdd(&accum_count[1], (unsigned long long)cnt);
  }
}

// ---------------------------------------------------------------------------
// Integer-pipe microbenchmark (roofline denominators, SURVEY 8d).  Eight
// independent dependency chains per thread, 1024 resident threads per SM.
// ---------------------------------------------------------------------------
template <int KIND>
__global__ void __launch_bounds__(256) microbench_kernel(unsigned *out, int iters, unsigned seed) {
  unsigned a[8];
  double d[8];
#pragma unroll
  for (int i = 0; i < 8; i++) {
    a[i] = seed * (threadIdx.x + 1) + i * 0x9e3779b9u;
    d[i] = (double)a[i] * 1e-9;
  }
  const unsigned b = seed | 0x01010101u, c = seed * 7u + 3u;
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int r = 0; r < 8; r++) {
#pragma unroll
      for (int i = 0; i < 8; i++) {  // opaque single instructions: no algebraic simplification
        if (KIND == 0) asm volatile("add.u32 %0, %0, %1;" : "+r"(a[i]) : "r"(b));
        else if (KIND == 1) asm volatile("mad.lo.u32 %0, %0, %1, %2;" : "+r"(a[i]) : "r"(b), "r"(c));
        else if (KIND == 2) asm volatile("vabsdiff4.u32.u32.u32.add %0, %1, %2, %0;" : "+r"(a[i]) : "r"(b), "r"(c));
        else if (KIND == 3) asm volatile("max.u16x2 %0, %0, %1;" : "+r"(a[i]) : "r"(b));
        else if (KIND == 4) asm volatile("dp4a.u32.u32 %0, %1, %2, %0;" : "+r"(a[i]) : "r"(b), "r"(c));
        else asm volatile("fma.rn.f64 %0, %0, %1, %2;" : "+d"(d[i]) : "d"(1.0000001), "d"(1e-9));
      }
    }
  }
  unsigned acc = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) acc += a[i] + (unsigned)(long long)d[i];
  if (acc == 0x12345678u) out[0] = acc;
}

}  // namespace tfk
