// Host side of libtf_gpu.so: the C ABI declared in include/tf_gpu.h.
//
// Mirrors what av1_temporal_filter() (av1/encoder/temporal_filter.c:1276-1312)
// does around the per-block loop: resolve the window into plain parameters,
// make the frames available to the workers (here: device frame cache with
// on-device border replication, the counterpart of av1_copy_and_extend_frame,
// av1/encoder/extend.c:113), run all blocks (here: one CUDA grid instead of
// the row job queue of av1/encoder/ethread.c:2062-2189), hand back the filtered
// frame and FRAME_DIFF.  No CPU fallback: without a CUDA device every entry
// point returns TF_GPU_ERR_NO_DEVICE.
#include "tf_kernels.cuh"
#include <cuda.h>  // CUdeviceptr / CUresult only; cuMemGetAddressRange is fetched through cudaGetDriverEntryPoint (no libcuda link)

#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#pragma GCC visibility push(default)
#include "../../include/tf_gpu.h"
#pragma GCC visibility pop

using namespace tfk;

namespace {

constexpr int DEV_BORDER = 80;  // luma device border (samples); see DESIGN.md "Data layout"

struct Geometry {
  int is_hbd, ss_x, ss_y, num_planes;
  int crop_w[2], crop_h[2], aligned_w[2], aligned_h[2];
  int bx[2], by[2], pitch[2], rows[2];
  bool operator==(const Geometry &o) const { return memcmp(this, &o, sizeof(*this)) == 0; }
};

struct DevFrame {
  uint64_t frame_id = 0;
  uint64_t last_use = 0;
  uint64_t pinned_epoch = 0;
  bool valid = false;
  Geometry g;
  void *base[3] = { nullptr, nullptr, nullptr };  // allocation base
  void *p00[3] = { nullptr, nullptr, nullptr };   // pixel (0,0)
  // cache slots only: luma row sums R16(i, j) = sum of Y(i, j + t), t < 16, with the luma pitch, for the lower bound
  // of the 16x16 search (rowsum16_kernel)
  uint16_t *rs_base = nullptr;
  uint16_t *rs00 = nullptr;  // at pixel (0,0)
  cudaEvent_t ready = nullptr;                    // upload + border extension + row sums finished (copy stream)
};

// Timing events of one filter call (main stream): start, after the search32 chain, after the
// search16 join, end.  One set per ticket and one for the resident path, so pipelined submits never
// read each other's times.
struct CallEvents {
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, evk[2] = { nullptr, nullptr };
};

struct Ticket {
  uint64_t id = 0;
  cudaEvent_t ev = nullptr;
  CallEvents te;
  int64_t *diff_dst = nullptr;
  bool want_diff = false;
  bool pending = false;
};

}  // namespace

struct tf_gpu_ctx {
  int device = 0;
  int num_sms = 148;
  cudaStream_t stream = nullptr;
  cudaStream_t stream2 = nullptr;  // 16x16 searches overlap the 32x32 chain
  cudaStream_t copy_stream = nullptr;  // uploads overlap the search of earlier frames
  cudaStream_t out_stream = nullptr;   // result read-back overlaps the search of the next window
  cudaEvent_t ev_out_ready = nullptr;  // output complete on the device (main stream)
  cudaEvent_t ev_out_done = nullptr;   // read-back of the device output finished (out stream)
  bool out_done_valid = false;
  // done_ev[e & 1] is recorded on the main stream at the end of call number e (every entry point that
  // takes a new epoch), so it also covers every earlier call; uploads into a cache slot wait for the
  // event that covers the call which used the slot last (see get_frame), not for the previous call,
  // so the next window's uploads overlap the current window's kernels.
  cudaEvent_t done_ev[2] = { nullptr, nullptr };
  bool done_valid[2] = { false, false };
  cudaEvent_t ev_f32[TF_GPU_MAX_FRAMES] = {};
  cudaEvent_t ev_s16 = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;   // microbenchmark and motion-search kernel timing
  CallEvents res_ev;                          // resident path
  const CallEvents *last_ev = nullptr;        // events of the last completed filter call
  bool split_valid = false;
  cudaStream_t noise_stream = nullptr;        // noise estimates do not queue behind a submitted window
  cudaEvent_t ev_async_upload = nullptr;      // last tf_gpu_cache_frame_async upload
  bool async_upload_pending = false;
  cudaEvent_t ev_ingest_src = nullptr;        // producer's stream at a tf_gpu_cache_frame_device call
  cudaEvent_t ev_search_src = nullptr;        // caller's stream at a tf_gpu_motion_search_device / tf_gpu_predict_device call
  cudaEvent_t ev_search_done = nullptr;       // that call's kernel on the main stream
  cudaEvent_t user_ev[4] = { nullptr, nullptr, nullptr, nullptr };
  std::vector<DevFrame> cache;
  DevFrame out;
  uint64_t use_counter = 0, epoch = 0;
  unsigned long long *d_diff = nullptr;   // [9][2]: one slot per ticket, slot 8 = resident path
  // slab mode over peer memory: another rank's output planes opened through CUDA IPC (tf_gpu_output_ipc_import)
  void *peer_base[3] = { nullptr, nullptr, nullptr };
  void *peer_out[3] = { nullptr, nullptr, nullptr };
  size_t peer_pitch[3] = { 0, 0, 0 };
  unsigned long long *h_diff = nullptr;   // pinned mirror
  unsigned long long *d_noise = nullptr;  // [2]
  unsigned long long *d_ctr = nullptr;    // [4] executed-work counters (instrumentation)
  unsigned long long h_ctr[4] = { 0, 0, 0, 0 };
  bool collect_counters = false;
  unsigned long long *h_noise = nullptr;
  Ticket tickets[8];
  uint64_t next_ticket = 1;
  int last_launches = 0;
  float last_kernel_ms = 0.f;
  // batched windows (tf_gpu_filter_batch_async): one output frame and one FRAME_DIFF slot per window, separate from
  // `out` and the ticket / resident slots; allocated by the first batch that needs them
  DevFrame bout[TF_GPU_MAX_BATCH];
  unsigned long long *d_bdiff = nullptr;  // [TF_GPU_MAX_BATCH][2]
  unsigned long long *h_bdiff = nullptr;  // pinned mirror
  int batch_n = 0;                        // windows of the last batch enqueued (0: none, or it failed)
  int batch_planes[TF_GPU_MAX_BATCH] = {}; // planes each window writes (its num_planes; bout[w] may hold more)
  CallEvents batch_ev;
  // dump buffers (device), grown on demand; 10, 11: full-pel search items / results, 12, 13: motion search
  void *d_dump[14] = {};
  size_t d_dump_sz[14] = {};
  char err[512] = { 0 };
};

namespace {

int fail(tf_gpu_ctx *c, int code, const char *fmt, ...) {
  if (c) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(c->err, sizeof(c->err), fmt, ap);
    va_end(ap);
  }
  return code;
}

#define CU(call)                                                                                     \
  do {                                                                                               \
    cudaError_t e_ = (call);                                                                         \
    if (e_ != cudaSuccess)                                                                           \
      return fail(ctx, e_ == cudaErrorMemoryAllocation ? TF_GPU_ERR_MEM : TF_GPU_ERR_CUDA, "%s: %s", \
                  #call, cudaGetErrorString(e_));                                                    \
  } while (0)

int align_up(int v, int a) { return (v + a - 1) / a * a; }

// Grid of a grid-stride kernel over n items: enough blocks for the items, at most `per_sm` per SM, at least one.
int grid_for(const tf_gpu_ctx *ctx, long long n, int threads, int per_sm) {
  long long b = (n + threads - 1) / threads;
  if (b > (long long)ctx->num_sms * per_sm) b = (long long)ctx->num_sms * per_sm;
  return b < 1 ? 1 : (int)b;
}

// Takes a new epoch for an entry point and records that epoch's completion event on the way out
// (also on error paths, so done_ev[e & 1] never refers to a call older than e - 2).
struct CallScope {
  tf_gpu_ctx *ctx;
  explicit CallScope(tf_gpu_ctx *c) : ctx(c) { ctx->epoch++; }
  ~CallScope() {
    const int i = (int)(ctx->epoch & 1);
    if (ctx->done_ev[i] && cudaEventRecord(ctx->done_ev[i], ctx->stream) == cudaSuccess) ctx->done_valid[i] = true;
  }
};

bool make_geometry(const tf_gpu_frame *f, int num_planes, Geometry *g, int luma_border = DEV_BORDER) {
  memset(g, 0, sizeof(*g));
  g->is_hbd = f->is_hbd ? 1 : 0;
  g->ss_x = f->ss_x;
  g->ss_y = f->ss_y;
  g->num_planes = num_planes;
  for (int k = 0; k < 2; k++) {
    g->crop_w[k] = f->crop_w[k];
    g->crop_h[k] = f->crop_h[k];
    g->aligned_w[k] = f->aligned_w[k];
    g->aligned_h[k] = f->aligned_h[k];
  }
  if (f->crop_w[0] <= 0 || f->crop_h[0] <= 0 || f->ss_x < 0 || f->ss_x > 1 || f->ss_y < 0 || f->ss_y > 1) return false;
  if (f->aligned_w[0] < f->crop_w[0] || f->aligned_h[0] < f->crop_h[0]) return false;
  for (int k = 0; k < 2; k++) {
    g->bx[k] = k ? luma_border >> f->ss_x : luma_border;
    g->by[k] = k ? luma_border >> f->ss_y : luma_border;
    g->pitch[k] = align_up(g->aligned_w[k] + 2 * g->bx[k], 128);
    g->rows[k] = g->aligned_h[k] + 2 * g->by[k] + 2;  // + slack rows: window / word over-reads stay inside
  }
  return true;
}

// cuMemGetAddressRange (allocation base and size of a device pointer), for the extent check of device frames
typedef CUresult (*AddressRangeFn)(CUdeviceptr *, size_t *, CUdeviceptr);
AddressRangeFn address_range_fn() {
  static AddressRangeFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void *p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuMemGetAddressRange", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = (AddressRangeFn)p;
  }
  return fn;
}
// `ptr` is device (or managed) memory of the context's device, `align`-byte aligned, and the `bytes` from it lie
// inside the allocation it belongs to.  Allocators that map memory in chunks (the virtual-memory API behind torch's
// expandable segments, stream-ordered pools) may report one chunk per call: the extent may go on into chunks mapped
// right after it, each device memory of this device, so the walk follows the ranges as long as they are contiguous.
// `what` names the pointer in the error message.
int check_device_extent(tf_gpu_ctx *ctx, const void *ptr, size_t bytes, size_t align, const char *what) {
  const AddressRangeFn range = address_range_fn();
  if (!range) return fail(ctx, TF_GPU_ERR_CUDA, "cuMemGetAddressRange is not available in this driver");
  if ((uintptr_t)ptr % align) return fail(ctx, TF_GPU_ERR_INVALID, "%s is not %zu-byte aligned", what, align);
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, ptr) != cudaSuccess) {
    cudaGetLastError();
    return fail(ctx, TF_GPU_ERR_INVALID, "%s is not a CUDA pointer", what);
  }
  if ((at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged) || at.device != ctx->device)
    return fail(ctx, TF_GPU_ERR_INVALID, "%s is not device memory of device %d", what, ctx->device);
  CUdeviceptr base = 0;
  size_t size = 0;
  const CUdeviceptr dp = (CUdeviceptr)(uintptr_t)ptr;
  if (range(&base, &size, dp) != CUDA_SUCCESS || dp < base || dp - base > size)
    return fail(ctx, TF_GPU_ERR_INVALID, "%s: no device allocation at this address", what);
  CUdeviceptr end = base + size;
  while (end - dp < bytes) {
    CUdeviceptr nb = 0;
    size_t ns = 0;
    cudaPointerAttributes na;
    if (range(&nb, &ns, end) != CUDA_SUCCESS || nb != end || ns == 0 ||
        cudaPointerGetAttributes(&na, (const void *)(uintptr_t)end) != cudaSuccess ||
        (na.type != cudaMemoryTypeDevice && na.type != cudaMemoryTypeManaged) || na.device != ctx->device) {
      cudaGetLastError();
      return fail(ctx, TF_GPU_ERR_INVALID, "%s: its extent (%zu bytes) runs past its allocation (%zu bytes)", what, bytes,
                  (size_t)(end - dp));
    }
    end = nb + ns;
  }
  return TF_GPU_OK;
}
// `rowsum`: the slot also gets the luma row-sum plane (frame cache slots; output frames do not).
int alloc_dev_frame(tf_gpu_ctx *ctx, DevFrame *d, const Geometry &g, bool rowsum = false) {
  const size_t es = g.is_hbd ? 2 : 1;
  if (d->base[0] && d->g == g && (!rowsum || d->rs_base)) return TF_GPU_OK;
  for (int p = 0; p < 3; p++) {
    if (d->base[p]) cudaFree(d->base[p]);
    d->base[p] = d->p00[p] = nullptr;
  }
  if (d->rs_base) cudaFree(d->rs_base);
  d->rs_base = d->rs00 = nullptr;
  d->g = g;
  d->valid = false;
  for (int p = 0; p < g.num_planes; p++) {
    const int k = p > 0;
    const size_t bytes = (size_t)g.rows[k] * g.pitch[k] * es;
    CU(cudaMalloc(&d->base[p], bytes));
    d->p00[p] = (char *)d->base[p] + ((size_t)g.by[k] * g.pitch[k] + g.bx[k]) * es;
  }
  if (rowsum) {
    CU(cudaMalloc(&d->rs_base, (size_t)g.rows[0] * g.pitch[0] * sizeof(uint16_t)));
    d->rs00 = d->rs_base + (size_t)g.by[0] * g.pitch[0] + g.bx[0];
  }
  return TF_GPU_OK;
}

// Row sums of a freshly filled slot's luma plane, on the copy stream before the slot's `ready` event: every column
// j of [-bx, aligned_w + bx - 16] and every row of [-by, aligned_h + by), the region a 16x16 candidate inside the
// MV limits can reach.  Part of filling the luma plane: last_launches keeps counting one launch per plane.
void launch_rowsum(tf_gpu_ctx *ctx, DevFrame *d) {
  const Geometry &g = d->g;
  const int w = g.aligned_w[0] + 2 * g.bx[0] - 15, h = g.aligned_h[0] + 2 * g.by[0];
  const dim3 grid((w + 16 * ROWSUM_THREADS - 1) / (16 * ROWSUM_THREADS), h);
  if (g.is_hbd)
    rowsum16_kernel<uint16_t><<<grid, ROWSUM_THREADS, 0, ctx->copy_stream>>>((const uint16_t *)d->p00[0], g.pitch[0],
                                                                             d->rs00, g.bx[0], g.by[0], w);
  else
    rowsum16_kernel<uint8_t><<<grid, ROWSUM_THREADS, 0, ctx->copy_stream>>>((const uint8_t *)d->p00[0], g.pitch[0],
                                                                            d->rs00, g.bx[0], g.by[0], w);
}

// Upload the crop area of a host frame and rebuild the borders on the device.
int upload_frame(tf_gpu_ctx *ctx, DevFrame *d, const tf_gpu_frame *f) {
  const Geometry &g = d->g;
  const size_t es = g.is_hbd ? 2 : 1;
  for (int p = 0; p < g.num_planes; p++) {
    const int k = p > 0;
    if (!f->plane[p]) return fail(ctx, TF_GPU_ERR_INVALID, "frame plane %d is NULL", p);
    CU(cudaMemcpy2DAsync(d->p00[p], (size_t)g.pitch[k] * es, f->plane[p], (size_t)f->stride[k] * es,
                         (size_t)g.crop_w[k] * es, g.crop_h[k], cudaMemcpyHostToDevice, ctx->copy_stream));
    const int ext_w = g.aligned_w[k] + g.bx[k], ext_h = g.aligned_h[k] + g.by[k];
    const long long n = (long long)g.crop_h[k] * (g.bx[k] + ext_w - g.crop_w[k]) + (long long)(g.by[k] + ext_h - g.crop_h[k]) * (g.bx[k] + ext_w);
    const int threads = 256;
    const int blocks = grid_for(ctx, n, threads, 16);
    if (g.is_hbd)
      extend_borders_kernel<uint16_t><<<blocks, threads, 0, ctx->copy_stream>>>((uint16_t *)d->p00[p], g.pitch[k],
                                                                          g.crop_w[k], g.crop_h[k], g.bx[k], g.by[k],
                                                                          ext_w, ext_h);
    else
      extend_borders_kernel<uint8_t><<<blocks, threads, 0, ctx->copy_stream>>>((uint8_t *)d->p00[p], g.pitch[k],
                                                                         g.crop_w[k], g.crop_h[k], g.bx[k], g.by[k],
                                                                         ext_w, ext_h);
    ctx->last_launches++;
  }
  launch_rowsum(ctx, d);
  CU(cudaGetLastError());
  CU(cudaEventRecord(d->ready, ctx->copy_stream));
  d->frame_id = f->frame_id;
  d->valid = true;
  return TF_GPU_OK;
}

// Fill a slot from device planes (tf_gpu_cache_frame_device, validated there): after the work already enqueued on
// the producer's stream, one ingest_plane_kernel per plane on the copy stream writes the same rectangle
// upload_frame() defines.
int ingest_frame(tf_gpu_ctx *ctx, DevFrame *d, const tf_gpu_frame *f, cudaStream_t src_stream) {
  const Geometry &g = d->g;
  CU(cudaEventRecord(ctx->ev_ingest_src, src_stream));
  CU(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_ingest_src, 0));
  for (int p = 0; p < g.num_planes; p++) {
    const int k = p > 0;
    const int ext_w = g.aligned_w[k] + g.bx[k], ext_h = g.aligned_h[k] + g.by[k];
    const int groups = (g.bx[k] + ext_w + (g.is_hbd ? 8 : 16) - 1) / (g.is_hbd ? 8 : 16);
    const dim3 grid((groups + INGEST_THREADS - 1) / INGEST_THREADS, (g.by[k] + ext_h + INGEST_ROWS - 1) / INGEST_ROWS);
    if (g.is_hbd)
      ingest_plane_kernel<uint16_t><<<grid, INGEST_THREADS, 0, ctx->copy_stream>>>(
          (uint16_t *)d->p00[p], g.pitch[k], (const uint16_t *)f->plane[p], f->stride[k], g.crop_w[k], g.crop_h[k],
          g.bx[k], g.by[k], ext_w, ext_h);
    else
      ingest_plane_kernel<uint8_t><<<grid, INGEST_THREADS, 0, ctx->copy_stream>>>(
          (uint8_t *)d->p00[p], g.pitch[k], (const uint8_t *)f->plane[p], f->stride[k], g.crop_w[k], g.crop_h[k],
          g.bx[k], g.by[k], ext_w, ext_h);
    ctx->last_launches++;
  }
  launch_rowsum(ctx, d);
  CU(cudaGetLastError());
  CU(cudaEventRecord(d->ready, ctx->copy_stream));
  d->frame_id = f->frame_id;
  d->valid = true;
  return TF_GPU_OK;
}

// Where a frame that is not resident comes from: the host (upload_frame) or device memory written on `stream`
// (ingest_frame).
struct FrameSource {
  bool device = false;
  cudaStream_t stream = nullptr;
};

DevFrame *find_cached(tf_gpu_ctx *ctx, uint64_t id, const Geometry *g) {
  if (!id) return nullptr;
  for (auto &d : ctx->cache)
    if (d.valid && d.frame_id == id && (!g || d.g == *g)) return &d;
  return nullptr;
}

// Returns a slot holding the frame (uploading if needed); the slot is pinned
// for the current epoch so that one window never evicts its own frames.
int get_frame(tf_gpu_ctx *ctx, const tf_gpu_frame *f, int num_planes, DevFrame **out,
              const FrameSource &src = FrameSource()) {
  Geometry g;
  if (!make_geometry(f, num_planes, &g)) return fail(ctx, TF_GPU_ERR_INVALID, "bad frame geometry");
  DevFrame *d = find_cached(ctx, f->frame_id, &g);
  if (!d) {
    // Victim choice, cheapest first: an allocated slot of the same geometry that holds nothing
    // (or an uncached scratch frame, id 0), then a never-allocated slot, then plain LRU.
    // Reusing allocations keeps cudaMalloc (device-synchronising) out of the steady state.
    DevFrame *victim = nullptr;
    int best_score = 99;
    for (auto &s : ctx->cache) {
      if (s.pinned_epoch == ctx->epoch) continue;
      const bool same = s.base[0] && s.g == g;
      int score;
      if (!s.valid && same) score = 0;
      else if (s.valid && s.frame_id == 0 && same) score = 1;
      else if (!s.valid) score = 2;
      else if (s.frame_id == 0) score = 3;
      else score = 4;
      if (s.pinned_epoch + 1 == ctx->epoch) score += 10;  // read by the call that may still be running: last resort
      if (score < best_score || (score == best_score && victim && s.last_use < victim->last_use)) {
        best_score = score;
        victim = &s;
      }
    }
    if (!victim) return fail(ctx, TF_GPU_ERR_MEM, "frame cache too small for this window");
    int rc = alloc_dev_frame(ctx, victim, g, true);
    if (rc) return rc;
    victim->valid = false;
    {
      // kernels of the call that used this slot last (epoch pinned_epoch) must have finished:
      // wait for the youngest recorded event that is not older than that call
      const int idx = (victim->pinned_epoch + 1 >= ctx->epoch) ? (int)((ctx->epoch - 1) & 1) : (int)(ctx->epoch & 1);
      if (victim->pinned_epoch > 0 && ctx->done_valid[idx])
        CU(cudaStreamWaitEvent(ctx->copy_stream, ctx->done_ev[idx], 0));
    }
    rc = src.device ? ingest_frame(ctx, victim, f, src.stream) : upload_frame(ctx, victim, f);
    if (rc) return rc;
    d = victim;
  }
  d->last_use = ++ctx->use_counter;
  d->pinned_epoch = ctx->epoch;
  *out = d;
  return TF_GPU_OK;
}

int validate_params(tf_gpu_ctx *ctx, const tf_gpu_params *p) {
  if (!p) return fail(ctx, TF_GPU_ERR_INVALID, "params is NULL");
  if (p->num_frames < 1 || p->num_frames > TF_GPU_MAX_FRAMES) return fail(ctx, TF_GPU_ERR_INVALID, "num_frames %d out of [1,%d]", p->num_frames, TF_GPU_MAX_FRAMES);
  if (p->filter_frame_idx < 0 || p->filter_frame_idx >= p->num_frames) return fail(ctx, TF_GPU_ERR_INVALID, "filter_frame_idx out of range");
  if (p->num_planes != 1 && p->num_planes != 3) return fail(ctx, TF_GPU_ERR_INVALID, "num_planes must be 1 or 3");
  if (p->bit_depth != 8 && p->bit_depth != 10 && p->bit_depth != 12) return fail(ctx, TF_GPU_ERR_INVALID, "bit_depth must be 8, 10 or 12");
  if (p->subpel_method < 0 || p->subpel_method > 2) return fail(ctx, TF_GPU_ERR_INVALID, "bad subpel_method");
  if (p->filter_strength < 0 || p->filter_strength > 6) return fail(ctx, TF_GPU_ERR_INVALID, "filter_strength out of [0,6]");
  if (p->q_factor < 0 || p->q_factor > 255 * 8) return fail(ctx, TF_GPU_ERR_INVALID, "q_factor out of range");
  if (p->subpel_iters_per_step < 1 || p->subpel_iters_per_step > 2) return fail(ctx, TF_GPU_ERR_INVALID, "subpel_iters_per_step must be 1 or 2");
  if (p->prune_mesh_level < 0 || p->prune_mesh_level > 2) return fail(ctx, TF_GPU_ERR_INVALID, "bad prune_mesh_level");
  for (int i = 0; i < 4; i++)
    if (p->mesh_patterns[i][0] < 0 || p->mesh_patterns[i][0] > 256 || p->mesh_patterns[i][1] < 0 || p->mesh_patterns[i][1] > 256)
      return fail(ctx, TF_GPU_ERR_INVALID, "mesh pattern %d out of [0,256]", i);
  // the smallest border the encoder configures is 64 (AOM_ENC_ALLINTRA_BORDER); below 40 the MV limits
  // of av1_set_mv_{row,col}_limits (mcomp.h:216-240) can invert
  if (p->border_in_pixels < 40 || p->border_in_pixels > 1024) return fail(ctx, TF_GPU_ERR_INVALID, "border_in_pixels out of [40,1024]");
  if (p->cm_width < 0 || p->cm_height < 0) return fail(ctx, TF_GPU_ERR_INVALID, "negative cm_width / cm_height");
  return TF_GPU_OK;
}

// Parameters against the geometry of the window: the device MV limits come from mi_rows / mi_cols while
// the device planes are sized from the frames' aligned size plus DEV_BORDER, so a caller whose mi grid
// exceeds the frames would make the search read outside the allocation.
int validate_geometry(tf_gpu_ctx *ctx, const tf_gpu_params *p, const Geometry &g) {
  if (p->mi_rows <= 0 || p->mi_cols <= 0) return fail(ctx, TF_GPU_ERR_INVALID, "mi_rows / mi_cols must be positive");
  // compared in mi units: the aligned sizes are multiples of 8, and mi_rows * 4 could overflow
  if (p->mi_rows > g.aligned_h[0] / 4 || p->mi_cols > g.aligned_w[0] / 4)
    return fail(ctx, TF_GPU_ERR_INVALID, "mi grid %dx%d (mi units) exceeds the frame's aligned size %dx%d", p->mi_cols,
                p->mi_rows, g.aligned_w[0], g.aligned_h[0]);
  if (g.is_hbd == 0 && p->bit_depth != 8) return fail(ctx, TF_GPU_ERR_INVALID, "8-bit container needs bit_depth 8");
  if (g.num_planes < p->num_planes) return fail(ctx, TF_GPU_ERR_INVALID, "frames lack chroma planes");
  return TF_GPU_OK;
}

void build_sites(Sites *s) {  // av1_init_motion_compensation_nstep (mcomp.c:433-475), level 0
  memset(s, 0, sizeof(*s));
  int radius = 1;
  for (int st = 0; st < 15; st++) {
    int tan_radius = (int)(0.41 * radius);
    if (tan_radius < 1) tan_radius = 1;
    int n = 12;
    if (radius <= 5) {
      tan_radius = radius;
      n = 8;
    }
    const int m[13][2] = { { 0, 0 },
                           { -radius, 0 },
                           { radius, 0 },
                           { 0, -radius },
                           { 0, radius },
                           { -radius, -tan_radius },
                           { radius, tan_radius },
                           { -tan_radius, radius },
                           { tan_radius, -radius },
                           { -radius, tan_radius },
                           { radius, -tan_radius },
                           { tan_radius, radius },
                           { -tan_radius, -radius } };
    for (int i = 0; i <= n; i++) {
      s->r[st][i] = (int16_t)m[i][0];
      s->c[st][i] = (int16_t)m[i][1];
    }
    s->n[st] = n;
    s->radius[st] = radius;
    if (st < 12) {
      const double a = radius * 1.5 + 0.5;
      radius = (int)(a > radius + 1 ? a : radius + 1);
    }
  }
}

const int16_t K12[16][12] = {  // av1_sub_pel_filters_12sharp, av1/common/filter.h:159-177
  { 0, 0, 0, 0, 0, 128, 0, 0, 0, 0, 0, 0 },         { 0, 1, -2, 3, -7, 127, 8, -4, 2, -1, 1, 0 },
  { -1, 2, -3, 6, -13, 124, 18, -8, 4, -2, 2, -1 }, { -1, 3, -4, 8, -18, 120, 28, -12, 7, -4, 2, -1 },
  { -1, 3, -6, 10, -21, 115, 38, -15, 8, -5, 3, -1 }, { -2, 4, -6, 12, -24, 108, 49, -18, 10, -6, 3, -2 },
  { -2, 4, -7, 13, -25, 100, 60, -21, 11, -7, 4, -2 }, { -2, 4, -7, 13, -26, 91, 71, -24, 13, -7, 4, -2 },
  { -2, 4, -7, 13, -25, 81, 81, -25, 13, -7, 4, -2 }, { -2, 4, -7, 13, -24, 71, 91, -26, 13, -7, 4, -2 },
  { -2, 4, -7, 11, -21, 60, 100, -25, 13, -7, 4, -2 }, { -2, 3, -6, 10, -18, 49, 108, -24, 12, -6, 4, -2 },
  { -1, 3, -5, 8, -15, 38, 115, -21, 10, -6, 3, -1 }, { -1, 2, -4, 7, -12, 28, 120, -18, 8, -4, 3, -1 },
  { -1, 2, -2, 4, -8, 18, 124, -13, 6, -3, 2, -1 },  { 0, 1, -1, 2, -4, 8, 127, -7, 3, -2, 1, 0 }
};
const int16_t K8[16][8] = {  // av1_sub_pel_filters_8, av1/common/filter.h:123-133
  { 0, 0, 0, 128, 0, 0, 0, 0 },      { 0, 2, -6, 126, 8, -2, 0, 0 },    { 0, 2, -10, 122, 18, -4, 0, 0 },
  { 0, 2, -12, 116, 28, -8, 2, 0 },  { 0, 2, -14, 110, 38, -10, 2, 0 }, { 0, 2, -14, 102, 48, -12, 2, 0 },
  { 0, 2, -16, 94, 58, -12, 2, 0 },  { 0, 2, -14, 84, 66, -12, 2, 0 },  { 0, 2, -14, 76, 76, -14, 2, 0 },
  { 0, 2, -12, 66, 84, -14, 2, 0 },  { 0, 2, -12, 58, 94, -16, 2, 0 },  { 0, 2, -12, 48, 102, -14, 2, 0 },
  { 0, 2, -10, 38, 110, -14, 2, 0 }, { 0, 2, -8, 28, 116, -12, 2, 0 },  { 0, 0, -4, 18, 122, -10, 2, 0 },
  { 0, 0, -2, 8, 126, -6, 2, 0 }
};

int ensure_dump(tf_gpu_ctx *ctx, int i, size_t bytes) {
  if (ctx->d_dump_sz[i] >= bytes) return TF_GPU_OK;
  if (ctx->d_dump[i]) cudaFree(ctx->d_dump[i]);
  ctx->d_dump[i] = nullptr;
  ctx->d_dump_sz[i] = 0;
  CU(cudaMalloc(&ctx->d_dump[i], bytes));
  ctx->d_dump_sz[i] = bytes;
  return TF_GPU_OK;
}

// Geometry, window and search parameters shared by every kernel (what tf_motion_search() and
// av1_tf_do_filtering_row() resolve from AV1_COMP before the per-block loop).
void fill_kparams(const tf_gpu_ctx *ctx, const tf_gpu_params *p, const Geometry &g, KParams &K) {
  memset(&K, 0, sizeof(K));
  K.width = g.crop_w[0];
  K.height = g.crop_h[0];
  K.mb_rows = (K.height + 31) / 32;  // get_num_blocks, temporal_filter.c:1236-1237
  K.mb_cols = (K.width + 31) / 32;
  K.mi_rows = p->mi_rows;
  K.mi_cols = p->mi_cols;
  K.ss_x = g.ss_x;
  K.ss_y = g.ss_y;
  K.num_planes = p->num_planes;
  K.bit_depth = p->bit_depth;
  K.is_hbd = g.is_hbd;
  for (int k = 0; k < 2; k++) {
    K.aligned_w[k] = g.aligned_w[k];
    K.aligned_h[k] = g.aligned_h[k];
    K.pitch[k] = g.pitch[k];
    K.out_pitch[k] = ctx->out.g.pitch[k];
  }
  K.border = p->border_in_pixels;
  K.num_frames = p->num_frames;
  K.filter_idx = p->filter_frame_idx;
  K.q_factor = p->q_factor;
  K.strength = p->filter_strength;
  K.force_integer_mv = p->force_integer_mv;
  K.allow_hp = p->allow_hp;
  K.subpel_method = p->subpel_method;
  K.iters_per_step = p->subpel_iters_per_step;
  K.prune_level = p->prune_mesh_level;
  for (int i = 0; i < 4; i++) {
    K.mesh[i][0] = p->mesh_patterns[i][0];
    K.mesh[i][1] = p->mesh_patterns[i][1];
  }
  K.use_skip = p->use_downsampled_sad ? 1 : 0;
  K.compute_diff = p->compute_frame_diff ? 1 : 0;
  // tf_motion_search() uses cm->width / cm->height (the coded size; temporal_filter.c:99-100)
  const int cm_w = p->cm_width > 0 ? p->cm_width : K.width, cm_h = p->cm_height > 0 ? p->cm_height : K.height;
  const int min_cm_size = cm_w < cm_h ? cm_w : cm_h;
  // MV_COST_L1_{LOW,MID,HD}RES (temporal_filter.c:119-122, mcomp.c:237-244)
  if (min_cm_size >= 720) { K.sad_lambda = 8; K.sse_lambda = 1; }
  else if (min_cm_size >= 480) { K.sad_lambda = 15; K.sse_lambda = 0; }
  else { K.sad_lambda = 32; K.sse_lambda = 2; }
  {  // av1_init_search_range (mcomp.c:217-226)
    int size = K.width > K.height ? K.width : K.height;
    if (size < 16) size = 16;
    int sr = 0;
    while ((size << sr) < 1023) sr++;
    K.step_param = sr < 9 ? sr : 9;
  }
  K.mse_thresh = ((min_cm_size >= 720) ? 12 : 3) << (p->bit_depth - 8);  // temporal_filter.c:249-250
  K.hbd_shift = g.is_hbd ? (p->bit_depth == 10 ? 2 : (p->bit_depth == 12 ? 4 : 0)) : 0;
}

// The KParams of one window writing into `out`, all rows: fill_kparams, the decay factors of the weights and the
// frame planes.  Shared by the single-window and the batched launches; each adds where its scratch and
// FRAME_DIFF go.
void window_kparams(const tf_gpu_ctx *ctx, const tf_gpu_params *p, DevFrame *const *frames, const Geometry &g,
                    const DevFrame &out, KParams &K) {
  fill_kparams(ctx, p, g, K);
  const int min_frame_size = K.width < K.height ? K.width : K.height;  // av1_apply_temporal_filter_c: the source size (:603)
  {  // decay factors, temporal_filter.c:583-597 (host libm, as the reference)
    double q_decay = pow((double)p->q_factor / 20, 2);
    q_decay = q_decay < 1e-5 ? 1e-5 : (q_decay > 1 ? 1 : q_decay);
    if (p->q_factor >= 128) q_decay = 0.5 * pow((double)p->q_factor / 64, 2);
    double s_decay = pow((double)p->filter_strength / 4, 2);
    s_decay = s_decay < 1e-5 ? 1e-5 : (s_decay > 1 ? 1 : s_decay);
    for (int pl = 0; pl < p->num_planes; pl++) {
      const double n_decay = 0.5 + log(2 * p->noise_levels[pl] + 5.0);
      K.decay[pl] = 1 / (n_decay * q_decay * s_decay);
    }
    double thr = min_frame_size * 0.1;  // TF_SEARCH_DISTANCE_THRESHOLD, :603-604
    K.dist_thr = thr > 1 ? thr : 1;
  }
  for (int f = 0; f < p->num_frames; f++)
    for (int pl = 0; pl < p->num_planes; pl++) K.frm[f][pl] = frames[f]->p00[pl];
  for (int f = 0; f < p->num_frames; f++) K.rs[f] = frames[f]->rs00;
  for (int k = 0; k < 2; k++) K.out_pitch[k] = out.g.pitch[k];
  for (int pl = 0; pl < p->num_planes; pl++) K.out[pl] = out.p00[pl];
  K.num_pels = 1024 + (p->num_planes > 1 ? 2 * (1024 >> (g.ss_x + g.ss_y)) : 0);
  K.row_begin = 0;
  K.row_end = K.mb_rows;
}

// Warps per SM of the denser register build of the 32x32 search (16-bit samples: 128 registers / 16 warps per SM,
// 1080p 10-bit 296 -> 310 frames/s; 8-bit: 96 / 20).
int s32_warps_hi(int is_hbd) { return is_hbd ? S32_WARPS_HI_HBD : S32_WARPS_HI; }

template <typename T, int MINB>
auto search32_kernel(const KParams &) { return tf_search32_kernel<T, MINB>; }
template <typename T, int MINB>
auto search32_kernel(const KParamsBatch &) { return tf_search32_batch_kernel<T, MINB>; }

// One launch of the 32x32 search on the main stream (KParamsBatch: the batched kernel).  The denser register build
// only where it saves a second wave: a grid that is resident at once with the 168-register build runs faster per
// block with it (no spills).
template <typename KP>
void launch_search32(const tf_gpu_ctx *ctx, int is_hbd, dim3 grid, const KP &K) {
  const long long blocks = (long long)grid.x * grid.y;
  const bool dense = blocks <= (long long)ctx->num_sms * s32_warps_hi(is_hbd) && blocks > (long long)ctx->num_sms * S32_WARPS_LO;
  if (is_hbd) {
    const auto kernel = dense ? search32_kernel<uint16_t, S32_WARPS_HI_HBD>(K) : search32_kernel<uint16_t, S32_WARPS_LO>(K);
    kernel<<<grid, 32, SearchSmem<uint16_t, 32>::TOTAL, ctx->stream>>>(K);
  } else {
    const auto kernel = dense ? search32_kernel<uint8_t, S32_WARPS_HI>(K) : search32_kernel<uint8_t, S32_WARPS_LO>(K);
    kernel<<<grid, 32, SearchSmem<uint8_t, 32>::TOTAL, ctx->stream>>>(K);
  }
}

// Build kernel parameters and launch the block kernel over rows [rb, re).
int launch_filter(tf_gpu_ctx *ctx, const tf_gpu_params *p, DevFrame *const *frames, const Geometry &g,
                  unsigned long long *d_diff, const tf_gpu_dump *dump, const CallEvents *te) {
  const bool timed = te != nullptr;
  KParams K;
  window_kparams(ctx, p, frames, g, ctx->out, K);
  for (int pl = 0; pl < p->num_planes; pl++) {
    if (ctx->peer_out[pl]) {  // the owner rank's plane: same geometry, hence the same pitch
      if (ctx->peer_pitch[pl] != (size_t)ctx->out.g.pitch[pl > 0] * (g.is_hbd ? 2 : 1))
        return fail(ctx, TF_GPU_ERR_INVALID, "imported output plane %d has a different pitch than this context's", pl);
      K.out[pl] = ctx->peer_out[pl];
    }
  }
  K.diff = d_diff;
  K.ctr = nullptr;
  if (ctx->collect_counters) {
    K.ctr = ctx->d_ctr;
    CU(cudaMemsetAsync(ctx->d_ctr, 0, 4 * sizeof(unsigned long long), ctx->stream));
  }
  if (p->out_row_end > p->out_row_begin) {
    K.row_begin = p->out_row_begin < 0 ? 0 : p->out_row_begin;
    K.row_end = p->out_row_end > K.mb_rows ? K.mb_rows : p->out_row_end;
  }
  const int nblocks_all = K.mb_rows * K.mb_cols;
  if (dump) {
    const size_t bf = (size_t)nblocks_all * p->num_frames;
    int rc = 0;
    if (dump->subblock_mvs) { rc = ensure_dump(ctx, 0, bf * 8 * sizeof(int16_t)); if (rc) return rc; K.d_mvs = (int16_t *)ctx->d_dump[0]; cudaMemsetAsync(K.d_mvs, 0, bf * 8 * sizeof(int16_t), ctx->stream); }
    if (dump->subblock_mses) { rc = ensure_dump(ctx, 1, bf * 4 * sizeof(int32_t)); if (rc) return rc; K.d_mses = (int32_t *)ctx->d_dump[1]; cudaMemsetAsync(K.d_mses, 0, bf * 4 * sizeof(int32_t), ctx->stream); }
    if (dump->pred) { rc = ensure_dump(ctx, 2, bf * K.num_pels * sizeof(uint16_t)); if (rc) return rc; K.d_pred = (uint16_t *)ctx->d_dump[2]; cudaMemsetAsync(K.d_pred, 0, bf * K.num_pels * sizeof(uint16_t), ctx->stream); }
    if (dump->accum) { rc = ensure_dump(ctx, 3, (size_t)nblocks_all * K.num_pels * sizeof(uint32_t)); if (rc) return rc; K.d_accum = (uint32_t *)ctx->d_dump[3]; }
    if (dump->count) { rc = ensure_dump(ctx, 4, (size_t)nblocks_all * K.num_pels * sizeof(uint16_t)); if (rc) return rc; K.d_count = (uint16_t *)ctx->d_dump[4]; }
  }
  {  // search results handed from the search kernels to the filter kernel
    const size_t bf = (size_t)nblocks_all * p->num_frames;
    int rc = ensure_dump(ctx, 5, bf * 2 * sizeof(int16_t));
    if (rc) return rc;
    rc = ensure_dump(ctx, 6, bf * sizeof(int32_t));
    if (rc) return rc;
    rc = ensure_dump(ctx, 7, bf * 8 * sizeof(int16_t));
    if (rc) return rc;
    rc = ensure_dump(ctx, 8, bf * 4 * sizeof(int32_t));
    if (rc) return rc;
    K.s_blk_mv = (int16_t *)ctx->d_dump[5];
    K.s_blk_mse = (int32_t *)ctx->d_dump[6];
    K.s_sub_mv = (int16_t *)ctx->d_dump[7];
    K.s_sub_mse = (int32_t *)ctx->d_dump[8];
    rc = ensure_dump(ctx, 9, (size_t)nblocks_all * 2 * sizeof(int16_t));
    if (rc) return rc;
    K.s_ref_mv = (int16_t *)ctx->d_dump[9];
  }
  const int grid = (K.row_end - K.row_begin) * K.mb_cols;
  if (grid <= 0) return fail(ctx, TF_GPU_ERR_INVALID, "empty row range");
  const size_t smem_filter = filter_smem_bytes(K.num_pels);
  const int nref = p->num_frames - 1;
  // the frame to filter is read by every kernel
  CU(cudaStreamWaitEvent(ctx->stream, frames[p->filter_frame_idx]->ready, 0));
  if (timed) CU(cudaEventRecord(te->ev0, ctx->stream));
  // Search phase: one search32 launch per reference frame on the main stream (the ref_mv
  // chain), the independent 16x16 searches of that frame on a second stream as soon as its
  // 32x32 results exist -> the throughput-bound 16x16 work fills the latency-bound chain.
  int nlaunch = 0;
  // Latency mode (a block-row slab of a frame whose blocks are resident at once): the per-frame launches make
  // every frame wait for the slowest block of the previous one although a block only depends on itself
  // (ref_mv); one search32 launch walks all frames of its block instead (time = the slowest block's total, not
  // the sum of the per-frame maxima), followed by one search16 launch over all frames.
  const bool row_range = (K.row_end - K.row_begin) < K.mb_rows;
  const bool fused_chain = nref > 0 && row_range && grid <= ctx->num_sms * s32_warps_hi(g.is_hbd);
  if (fused_chain) {
    for (int f = 0; f < p->num_frames; f++)
      if (f != p->filter_frame_idx) CU(cudaStreamWaitEvent(ctx->stream, frames[f]->ready, 0));
    KParams Kf = K;
    Kf.frame_begin = 0;
    Kf.frame_end = p->num_frames;
    launch_search32(ctx, g.is_hbd, grid, Kf);
    nlaunch++;
    if (timed) cudaEventRecord(te->evk[0], ctx->stream);
    if (!p->force_integer_mv) {
      if (g.is_hbd) tf_search16_kernel<uint16_t><<<grid * 4 * nref, 32, SearchSmem<uint16_t, 16>::TOTAL, ctx->stream>>>(Kf);
      else tf_search16_kernel<uint8_t><<<grid * 4 * nref, 32, SearchSmem<uint8_t, 16>::TOTAL, ctx->stream>>>(Kf);
      nlaunch++;
    }
    if (timed) cudaEventRecord(te->evk[1], ctx->stream);
  } else if (nref > 0) {
    // (Measured and rejected: one search16 launch over all frames after the chain instead: 4K 10-bit with three
    // windows in flight 62.6 -> 63.6 frames/s, 1080p 329 -> 321, and a single window loses the overlap with its own
    // chain.)
    for (int f = 0; f < p->num_frames; f++) {
      if (f == p->filter_frame_idx) continue;
      KParams Kf = K;
      Kf.frame_begin = f;
      Kf.frame_end = f + 1;
      if (f > 0 && f - 1 == p->filter_frame_idx) Kf.frame_begin = f - 1;  // negate ref_mv at the centre frame
      CU(cudaStreamWaitEvent(ctx->stream, frames[f]->ready, 0));  // uploads of later frames overlap this search
      launch_search32(ctx, g.is_hbd, grid, Kf);
      nlaunch++;
      if (!p->force_integer_mv) {
        CU(cudaEventRecord(ctx->ev_f32[f], ctx->stream));
        CU(cudaStreamWaitEvent(ctx->stream2, ctx->ev_f32[f], 0));
        Kf.frame_begin = f;
        Kf.frame_end = f + 1;
        KParams K16 = Kf;
        // task decode expects [frame_begin, frame_end) minus the centre: a single non-centre frame
        K16.filter_idx = K.filter_idx;
        if (g.is_hbd) tf_search16_kernel<uint16_t><<<grid * 4, 32, SearchSmem<uint16_t, 16>::TOTAL, ctx->stream2>>>(K16);
        else tf_search16_kernel<uint8_t><<<grid * 4, 32, SearchSmem<uint8_t, 16>::TOTAL, ctx->stream2>>>(K16);
        nlaunch++;
      }
    }
    if (timed) cudaEventRecord(te->evk[0], ctx->stream);
    if (!p->force_integer_mv) {
      CU(cudaEventRecord(ctx->ev_s16, ctx->stream2));
      CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_s16, 0));
    }
    if (timed) cudaEventRecord(te->evk[1], ctx->stream);
  }
  // the filter kernel overwrites the device output: the previous call's read-back must be over
  if (ctx->out_done_valid) CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_out_done, 0));
  if (g.is_hbd) tf_filter_kernel<uint16_t><<<grid, FILT_THREADS, smem_filter, ctx->stream>>>(K);
  else tf_filter_kernel<uint8_t><<<grid, FILT_THREADS, smem_filter, ctx->stream>>>(K);
  nlaunch++;
  CU(cudaGetLastError());
  if (timed) CU(cudaEventRecord(te->ev1, ctx->stream));
  ctx->last_launches += nlaunch - 1;
  ctx->split_valid = timed && nref > 0;
  if (timed) ctx->last_ev = te;
  ctx->last_launches++;
  return TF_GPU_OK;
}

// The batched form of launch_filter: n windows over one geometry, every block row, each window into its own
// output frame (ctx->bout[w]) and FRAME_DIFF slot.  Three launches on the main stream: the fused 32x32 chain
// (every frame of a (window, block) in one warp) over the windows that have a reference frame, the 16x16 tasks over
// the windows that have any, the filter over all.  Each kernel gets only the windows that have work for it, so
// grid y never holds a window whose blocks would all exit.
int launch_filter_batch(tf_gpu_ctx *ctx, int n, const tf_gpu_params *params,
                        DevFrame *const (*frames)[TF_GPU_MAX_FRAMES], const Geometry &g, const CallEvents *te) {
  const int mb_cols = (g.crop_w[0] + 31) / 32, nblk = ((g.crop_h[0] + 31) / 32) * mb_cols;
  // search scratch: window w's [blocks][num_frames] slices follow those of the windows before it
  size_t bf_total = 0;
  for (int w = 0; w < n; w++) bf_total += (size_t)nblk * params[w].num_frames;
  int rc = ensure_dump(ctx, 5, bf_total * 2 * sizeof(int16_t));
  if (!rc) rc = ensure_dump(ctx, 6, bf_total * sizeof(int32_t));
  if (!rc) rc = ensure_dump(ctx, 7, bf_total * 8 * sizeof(int16_t));
  if (!rc) rc = ensure_dump(ctx, 8, bf_total * 4 * sizeof(int32_t));
  if (!rc) rc = ensure_dump(ctx, 9, (size_t)n * nblk * 2 * sizeof(int16_t));
  if (rc) return rc;
  KParamsBatch all, s32, s16;
  int n32 = 0, n16 = 0, max_nref16 = 0, max_pels = 0;
  size_t bf = 0;
  for (int w = 0; w < n; w++) {
    const tf_gpu_params *p = &params[w];
    KParams &K = all.w[w];
    window_kparams(ctx, p, frames[w], g, ctx->bout[w], K);
    K.diff = ctx->d_bdiff + 2 * w;
    K.s_blk_mv = (int16_t *)ctx->d_dump[5] + bf * 2;
    K.s_blk_mse = (int32_t *)ctx->d_dump[6] + bf;
    K.s_sub_mv = (int16_t *)ctx->d_dump[7] + bf * 8;
    K.s_sub_mse = (int32_t *)ctx->d_dump[8] + bf * 4;
    K.s_ref_mv = (int16_t *)ctx->d_dump[9] + (size_t)w * nblk * 2;
    K.frame_begin = 0;
    K.frame_end = p->num_frames;
    bf += (size_t)nblk * p->num_frames;
    if (K.num_pels > max_pels) max_pels = K.num_pels;
    const int nref = p->num_frames - 1;
    if (nref > 0) {  // the same rules as launch_filter: no reference frame, no search; integer MVs, no 16x16 search
      s32.w[n32++] = K;
      if (!p->force_integer_mv) {
        s16.w[n16++] = K;
        if (nref > max_nref16) max_nref16 = nref;
      }
    }
  }
  CU(cudaMemsetAsync(ctx->d_bdiff, 0, (size_t)n * 2 * sizeof(unsigned long long), ctx->stream));
  CU(cudaEventRecord(te->ev0, ctx->stream));
  int nlaunch = 0;
  if (n32) {
    launch_search32(ctx, g.is_hbd, dim3(nblk, n32), s32);  // the register build from the grid of the whole batch
    nlaunch++;
  }
  CU(cudaEventRecord(te->evk[0], ctx->stream));
  if (n16) {
    const dim3 grid(nblk * 4 * max_nref16, n16);
    if (g.is_hbd) tf_search16_batch_kernel<uint16_t><<<grid, 32, SearchSmem<uint16_t, 16>::TOTAL, ctx->stream>>>(s16);
    else tf_search16_batch_kernel<uint8_t><<<grid, 32, SearchSmem<uint8_t, 16>::TOTAL, ctx->stream>>>(s16);
    nlaunch++;
  }
  CU(cudaEventRecord(te->evk[1], ctx->stream));
  const dim3 grid(nblk, n);
  if (g.is_hbd) tf_filter_batch_kernel<uint16_t><<<grid, FILT_THREADS, filter_smem_bytes(max_pels), ctx->stream>>>(all);
  else tf_filter_batch_kernel<uint8_t><<<grid, FILT_THREADS, filter_smem_bytes(max_pels), ctx->stream>>>(all);
  nlaunch++;
  CU(cudaGetLastError());
  CU(cudaEventRecord(te->ev1, ctx->stream));
  ctx->last_launches += nlaunch;
  ctx->split_valid = n32 > 0;
  ctx->last_ev = te;
  return TF_GPU_OK;
}

int download_dump(tf_gpu_ctx *ctx, const tf_gpu_params *p, const Geometry &g, const tf_gpu_dump *dump) {
  const int mb_rows = (g.crop_h[0] + 31) / 32, mb_cols = (g.crop_w[0] + 31) / 32;
  const size_t nb = (size_t)mb_rows * mb_cols, bf = nb * p->num_frames;
  const int num_pels = 1024 + (p->num_planes > 1 ? 2 * (1024 >> (g.ss_x + g.ss_y)) : 0);
  if (dump->subblock_mvs) CU(cudaMemcpyAsync(dump->subblock_mvs, ctx->d_dump[0], bf * 8 * sizeof(int16_t), cudaMemcpyDeviceToHost, ctx->stream));
  if (dump->subblock_mses) CU(cudaMemcpyAsync(dump->subblock_mses, ctx->d_dump[1], bf * 4 * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
  if (dump->pred) CU(cudaMemcpyAsync(dump->pred, ctx->d_dump[2], bf * num_pels * sizeof(uint16_t), cudaMemcpyDeviceToHost, ctx->stream));
  if (dump->accum) CU(cudaMemcpyAsync(dump->accum, ctx->d_dump[3], nb * num_pels * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  if (dump->count) CU(cudaMemcpyAsync(dump->count, ctx->d_dump[4], nb * num_pels * sizeof(uint16_t), cudaMemcpyDeviceToHost, ctx->stream));
  return TF_GPU_OK;
}

// Copy block rows [rb, re) of the first num_planes planes of a device output frame (ctx->out or a batch output)
// into the caller's planes (num_planes < 0: all planes of the frame).
int download_rows(tf_gpu_ctx *ctx, const DevFrame &dev, tf_gpu_frame *out, int rb, int re, cudaStream_t os,
                  int num_planes = -1) {
  const Geometry &g = dev.g;
  const size_t es = g.is_hbd ? 2 : 1;
  const int mb_cols = (g.crop_w[0] + 31) / 32;
  const int np = num_planes < 0 || num_planes > g.num_planes ? g.num_planes : num_planes;
  for (int pl = 0; pl < np; pl++) {
    const int k = pl > 0;
    const int bh = 32 >> (pl ? g.ss_y : 0), bw = 32 >> (pl ? g.ss_x : 0);
    if (!out->plane[pl]) return fail(ctx, TF_GPU_ERR_INVALID, "output plane %d is NULL", pl);
    // full blocks, as temporal_filter.c:740-777 writes them, but never beyond the
    // host allocation (aligned size + host border)
    int cols = mb_cols * bw, y0 = rb * bh, y1 = re * bh;
    const int max_cols = out->aligned_w[k] + (k ? out->border >> g.ss_x : out->border);
    const int max_rows = out->aligned_h[k] + (k ? out->border >> g.ss_y : out->border);
    if (cols > max_cols) cols = max_cols;
    if (cols > out->stride[k]) cols = out->stride[k];
    if (y1 > max_rows) y1 = max_rows;
    if (y1 <= y0) continue;
    char *dst = (char *)out->plane[pl] + (size_t)y0 * out->stride[k] * es;
    const char *src = (const char *)dev.p00[pl] + (size_t)y0 * g.pitch[k] * es;
    CU(cudaMemcpy2DAsync(dst, (size_t)out->stride[k] * es, src, (size_t)g.pitch[k] * es, (size_t)cols * es, y1 - y0,
                         cudaMemcpyDeviceToHost, os));
  }
  return TF_GPU_OK;
}

// aom_extend_frame_borders_c (aom_scale/generic/yv12extend.c:183-223) on the device output, then the
// whole extended allocation (host border on every side) goes back in one 2-D copy per plane.
int extend_and_download_output(tf_gpu_ctx *ctx, tf_gpu_frame *out, cudaStream_t os) {
  const Geometry &g = ctx->out.g;
  const size_t es = g.is_hbd ? 2 : 1;
  for (int pl = 0; pl < g.num_planes; pl++) {
    const int k = pl > 0;
    const int hb_x = k ? out->border >> g.ss_x : out->border, hb_y = k ? out->border >> g.ss_y : out->border;
    const int ext_w = g.aligned_w[k] + hb_x, ext_h = g.aligned_h[k] + hb_y;  // right / bottom extents from pixel 0
    const long long n = (long long)g.crop_h[k] * (hb_x + ext_w - g.crop_w[k]) + (long long)(hb_y + ext_h - g.crop_h[k]) * (hb_x + ext_w);
    const int threads = 256;
    const int blocks = grid_for(ctx, n, threads, 16);
    if (!out->plane[pl]) return fail(ctx, TF_GPU_ERR_INVALID, "output plane %d is NULL", pl);
    if (g.is_hbd)
      extend_borders_kernel<uint16_t><<<blocks, threads, 0, ctx->stream>>>((uint16_t *)ctx->out.p00[pl], g.pitch[k], g.crop_w[k], g.crop_h[k], hb_x, hb_y, ext_w, ext_h);
    else
      extend_borders_kernel<uint8_t><<<blocks, threads, 0, ctx->stream>>>((uint8_t *)ctx->out.p00[pl], g.pitch[k], g.crop_w[k], g.crop_h[k], hb_x, hb_y, ext_w, ext_h);
    ctx->last_launches++;
  }
  CU(cudaGetLastError());
  if (os != ctx->stream) {
    CU(cudaEventRecord(ctx->ev_out_ready, ctx->stream));
    CU(cudaStreamWaitEvent(os, ctx->ev_out_ready, 0));
  }
  for (int pl = 0; pl < g.num_planes; pl++) {
    const int k = pl > 0;
    const int hb_x = k ? out->border >> g.ss_x : out->border, hb_y = k ? out->border >> g.ss_y : out->border;
    const int ext_w = g.aligned_w[k] + hb_x, ext_h = g.aligned_h[k] + hb_y;
    char *dst = (char *)out->plane[pl] - ((size_t)hb_y * out->stride[k] + hb_x) * es;
    const char *src = (const char *)ctx->out.p00[pl] - ((size_t)hb_y * g.pitch[k] + hb_x) * es;
    CU(cudaMemcpy2DAsync(dst, (size_t)out->stride[k] * es, src, (size_t)g.pitch[k] * es, (size_t)(hb_x + ext_w) * es,
                         hb_y + ext_h, cudaMemcpyDeviceToHost, os));
  }
  return TF_GPU_OK;
}

// Pointer, pitch and full-block extent of a plane of a device output frame.
void device_plane(const DevFrame &d, int plane, void **dptr, size_t *pitch_bytes, int *rows, int *row_bytes) {
  const Geometry &g = d.g;
  const int k = plane > 0;
  const size_t es = g.is_hbd ? 2 : 1;
  if (dptr) *dptr = d.p00[plane];
  if (pitch_bytes) *pitch_bytes = (size_t)g.pitch[k] * es;
  if (rows) *rows = ((g.crop_h[0] + 31) / 32) * (32 >> (plane ? g.ss_y : 0));
  if (row_bytes) *row_bytes = (int)(((g.crop_w[0] + 31) / 32) * (32 >> (plane ? g.ss_x : 0)) * es);
}

int submit_impl(tf_gpu_ctx *ctx, const tf_gpu_params *params, const tf_gpu_frame *frames, tf_gpu_frame *out,
                int64_t diff_sum_sse[2], const tf_gpu_dump *dump, uint64_t *ticket_out) {
  if (!ctx) return TF_GPU_ERR_INVALID;
  int rc = validate_params(ctx, params);
  if (rc) return rc;
  if (!frames || !out) return fail(ctx, TF_GPU_ERR_INVALID, "frames/out is NULL");
  CU(cudaSetDevice(ctx->device));
  if ((int)ctx->cache.size() < params->num_frames) return fail(ctx, TF_GPU_ERR_MEM, "frame cache smaller than the window");
  CallScope scope(ctx);
  ctx->last_launches = 0;
  DevFrame *devf[TF_GPU_MAX_FRAMES];
  // upload order = consumption order: the frame to filter first, then the chain order
  for (int k = 0; k < params->num_frames; k++) {
    const int i = k == 0 ? params->filter_frame_idx : (k <= params->filter_frame_idx ? k - 1 : k);
    if (frames[i].is_hbd != frames[0].is_hbd) return fail(ctx, TF_GPU_ERR_INVALID, "mixed bit depth containers");
    rc = get_frame(ctx, &frames[i], params->num_planes, &devf[i]);
    if (rc) return rc;
  }
  for (int i = 0; i < params->num_frames; i++)
    if (!(devf[i]->g == devf[0]->g)) return fail(ctx, TF_GPU_ERR_INVALID, "frames of one window must share geometry");
  const Geometry &g = devf[0]->g;
  rc = validate_geometry(ctx, params, g);
  if (rc) return rc;
  if (ctx->peer_out[0] || ctx->peer_out[1] || ctx->peer_out[2])
    return fail(ctx, TF_GPU_ERR_INVALID, "an output plane is imported from another rank: its rows go there, use the resident calls");
  Geometry og = g;
  const bool extend_out = params->extend_output_borders && !(params->out_row_end > params->out_row_begin);
  if (extend_out) {
    // the output frame carries the host's full border so the extended allocation can be returned
    const int ob = ((out->border > DEV_BORDER ? out->border : DEV_BORDER) + 15) & ~15;
    if (!make_geometry(out, params->num_planes, &og, ob)) return fail(ctx, TF_GPU_ERR_INVALID, "bad output geometry");
    if (!(og.crop_w[0] == g.crop_w[0] && og.crop_h[0] == g.crop_h[0] && og.is_hbd == g.is_hbd && og.ss_x == g.ss_x && og.ss_y == g.ss_y))
      return fail(ctx, TF_GPU_ERR_INVALID, "output frame does not match the window geometry");
    for (int k = 0; k < 2; k++)
      if (out->stride[k] < og.aligned_w[k] + 2 * (k ? out->border >> og.ss_x : out->border))
        return fail(ctx, TF_GPU_ERR_INVALID, "output stride too small for its border");
  }
  rc = alloc_dev_frame(ctx, &ctx->out, og);
  if (rc) return rc;
  Ticket &t = ctx->tickets[ctx->next_ticket % 8];
  if (t.pending) return fail(ctx, TF_GPU_ERR_INVALID, "too many submits in flight (max 8)");
  const int slot = (int)(ctx->next_ticket % 8);
  unsigned long long *d_diff = ctx->d_diff + 2 * slot;
  CU(cudaMemsetAsync(d_diff, 0, 2 * sizeof(unsigned long long), ctx->stream));
  rc = launch_filter(ctx, params, devf, g, d_diff, dump, &t.te);
  if (rc) return rc;
  const int mb_rows = (g.crop_h[0] + 31) / 32;
  int rb = 0, re = mb_rows;
  if (params->out_row_end > params->out_row_begin) {
    rb = params->out_row_begin < 0 ? 0 : params->out_row_begin;
    re = params->out_row_end > mb_rows ? mb_rows : params->out_row_end;
  }
  // the result goes back on its own stream so that the next window's search is not held up by
  // the copy (debug dumps keep everything on the main stream)
  cudaStream_t os = dump ? ctx->stream : ctx->out_stream;
  if (extend_out) {
    rc = extend_and_download_output(ctx, out, os);
    if (rc) return rc;
  } else {
    if (os != ctx->stream) {
      CU(cudaEventRecord(ctx->ev_out_ready, ctx->stream));
      CU(cudaStreamWaitEvent(os, ctx->ev_out_ready, 0));
    }
    rc = download_rows(ctx, ctx->out, out, rb, re, os);
    if (rc) return rc;
  }
  if (dump) {
    rc = download_dump(ctx, params, g, dump);
    if (rc) return rc;
  }
  CU(cudaMemcpyAsync(ctx->h_diff + 2 * slot, d_diff, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, os));
  CU(cudaEventRecord(t.ev, os));
  if (os != ctx->stream) {
    CU(cudaEventRecord(ctx->ev_out_done, os));
    ctx->out_done_valid = true;
  }
  t.id = ctx->next_ticket++;
  t.diff_dst = diff_sum_sse;
  t.want_diff = diff_sum_sse != nullptr;
  t.pending = true;
  *ticket_out = t.id;
  return TF_GPU_OK;
}

}  // namespace

extern "C" {

int tf_gpu_abi_version(void) { return TF_GPU_ABI_VERSION; }

int tf_gpu_create(tf_gpu_ctx **out, const tf_gpu_device_cfg *cfg) {
  if (!out) return TF_GPU_ERR_INVALID;
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) return TF_GPU_ERR_NO_DEVICE;
  tf_gpu_ctx *ctx = new (std::nothrow) tf_gpu_ctx();
  if (!ctx) return TF_GPU_ERR_MEM;
  int dev = cfg ? cfg->device : -1;
  if (dev < 0) {
    if (cudaGetDevice(&dev) != cudaSuccess) dev = 0;
  }
  if (dev >= ndev) {
    delete ctx;
    return TF_GPU_ERR_NO_DEVICE;
  }
  ctx->device = dev;
  {
    int sms = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && sms > 0) ctx->num_sms = sms;
  }
  int slots = (cfg && cfg->max_cached_frames > 0) ? cfg->max_cached_frames : 32;
  if (slots < TF_GPU_MAX_FRAMES) slots = TF_GPU_MAX_FRAMES;
  ctx->cache.resize(slots);
  cudaError_t e = cudaSetDevice(dev);
  // the ref_mv chain on the main stream is the critical path: give it priority over the
  // independent 16x16 searches that fill the machine underneath it
  int prio_lo = 0, prio_hi = 0;
  if (e == cudaSuccess) e = cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
  if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&ctx->stream, cudaStreamNonBlocking, prio_hi);
  if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&ctx->stream2, cudaStreamNonBlocking, prio_lo);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->out_stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_out_ready, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_out_done, cudaEventDisableTiming);
  for (int i = 0; i < 2; i++)
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->done_ev[i], cudaEventDisableTiming);
  for (auto &d : ctx->cache)
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&d.ready, cudaEventDisableTiming);
  for (int i = 0; i < TF_GPU_MAX_FRAMES && e == cudaSuccess; i++) e = cudaEventCreateWithFlags(&ctx->ev_f32[i], cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_s16, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreate(&ctx->ev0);
  if (e == cudaSuccess) e = cudaEventCreate(&ctx->ev1);
  auto make_call_events = [&](CallEvents &te) {
    if (e == cudaSuccess) e = cudaEventCreate(&te.ev0);
    if (e == cudaSuccess) e = cudaEventCreate(&te.ev1);
    if (e == cudaSuccess) e = cudaEventCreate(&te.evk[0]);
    if (e == cudaSuccess) e = cudaEventCreate(&te.evk[1]);
  };
  make_call_events(ctx->res_ev);
  make_call_events(ctx->batch_ev);
  for (int i = 0; i < 8; i++) make_call_events(ctx->tickets[i].te);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->noise_stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_async_upload, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_ingest_src, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_search_src, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_search_done, cudaEventDisableTiming);
  for (int i = 0; i < 4 && e == cudaSuccess; i++) e = cudaEventCreate(&ctx->user_ev[i]);
  for (int i = 0; i < 8 && e == cudaSuccess; i++) e = cudaEventCreateWithFlags(&ctx->tickets[i].ev, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaMalloc(&ctx->d_diff, 18 * sizeof(unsigned long long));
  if (e == cudaSuccess) e = cudaMallocHost(&ctx->h_diff, 18 * sizeof(unsigned long long));
  if (e == cudaSuccess) e = cudaMalloc(&ctx->d_noise, 2 * sizeof(unsigned long long));
  if (e == cudaSuccess) e = cudaMalloc(&ctx->d_ctr, 4 * sizeof(unsigned long long));
  if (e == cudaSuccess) e = cudaMallocHost(&ctx->h_noise, 2 * sizeof(unsigned long long));
  if (e == cudaSuccess) {
    Sites s;
    build_sites(&s);
    e = cudaMemcpyToSymbol(c_sites, &s, sizeof(s));
  }
  if (e == cudaSuccess) e = cudaMemcpyToSymbol(c_k12, K12, sizeof(K12));
  if (e == cudaSuccess) e = cudaMemcpyToSymbol(c_k8, K8, sizeof(K8));
  if (e == cudaSuccess) e = cudaFuncSetAttribute(tf_filter_kernel<uint8_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)filter_smem_bytes(3072));
  if (e == cudaSuccess) e = cudaFuncSetAttribute(tf_filter_kernel<uint16_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)filter_smem_bytes(3072));
  if (e == cudaSuccess) e = cudaFuncSetAttribute(tf_filter_batch_kernel<uint8_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)filter_smem_bytes(3072));
  if (e == cudaSuccess) e = cudaFuncSetAttribute(tf_filter_batch_kernel<uint16_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)filter_smem_bytes(3072));
  if (e != cudaSuccess) {
    tf_gpu_destroy(ctx);
    return e == cudaErrorMemoryAllocation ? TF_GPU_ERR_MEM : TF_GPU_ERR_CUDA;
  }
  *out = ctx;
  return TF_GPU_OK;
}

void tf_gpu_destroy(tf_gpu_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
  if (ctx->out_stream) cudaStreamSynchronize(ctx->out_stream);
  for (auto &d : ctx->cache) {
    for (int p = 0; p < 3; p++)
      if (d.base[p]) cudaFree(d.base[p]);
    if (d.rs_base) cudaFree(d.rs_base);
    if (d.ready) cudaEventDestroy(d.ready);
  }
  for (int i = 0; i < 2; i++)
    if (ctx->done_ev[i]) cudaEventDestroy(ctx->done_ev[i]);
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  if (ctx->out_stream) cudaStreamDestroy(ctx->out_stream);
  if (ctx->ev_out_ready) cudaEventDestroy(ctx->ev_out_ready);
  if (ctx->ev_out_done) cudaEventDestroy(ctx->ev_out_done);
  for (int p = 0; p < 3; p++)
    if (ctx->out.base[p]) cudaFree(ctx->out.base[p]);
  for (auto &b : ctx->bout)
    for (int p = 0; p < 3; p++)
      if (b.base[p]) cudaFree(b.base[p]);
  if (ctx->d_bdiff) cudaFree(ctx->d_bdiff);
  if (ctx->h_bdiff) cudaFreeHost(ctx->h_bdiff);
  for (int i = 0; i < (int)(sizeof(ctx->d_dump) / sizeof(ctx->d_dump[0])); i++)
    if (ctx->d_dump[i]) cudaFree(ctx->d_dump[i]);
  for (int p = 0; p < 3; p++)
    if (ctx->peer_base[p]) cudaIpcCloseMemHandle(ctx->peer_base[p]);
  if (ctx->d_diff) cudaFree(ctx->d_diff);
  if (ctx->h_diff) cudaFreeHost(ctx->h_diff);
  if (ctx->d_noise) cudaFree(ctx->d_noise);
  if (ctx->d_ctr) cudaFree(ctx->d_ctr);
  if (ctx->h_noise) cudaFreeHost(ctx->h_noise);
  for (int i = 0; i < 8; i++)
    if (ctx->tickets[i].ev) cudaEventDestroy(ctx->tickets[i].ev);
  for (int i = 0; i < 4; i++)
    if (ctx->user_ev[i]) cudaEventDestroy(ctx->user_ev[i]);
  auto drop_call_events = [](CallEvents &te) {
    if (te.ev0) cudaEventDestroy(te.ev0);
    if (te.ev1) cudaEventDestroy(te.ev1);
    if (te.evk[0]) cudaEventDestroy(te.evk[0]);
    if (te.evk[1]) cudaEventDestroy(te.evk[1]);
  };
  drop_call_events(ctx->res_ev);
  drop_call_events(ctx->batch_ev);
  for (int i = 0; i < 8; i++) drop_call_events(ctx->tickets[i].te);
  if (ctx->noise_stream) {
    cudaStreamSynchronize(ctx->noise_stream);
    cudaStreamDestroy(ctx->noise_stream);
  }
  if (ctx->ev_async_upload) cudaEventDestroy(ctx->ev_async_upload);
  if (ctx->ev_ingest_src) cudaEventDestroy(ctx->ev_ingest_src);
  if (ctx->ev_search_src) cudaEventDestroy(ctx->ev_search_src);
  if (ctx->ev_search_done) cudaEventDestroy(ctx->ev_search_done);
  if (ctx->ev0) cudaEventDestroy(ctx->ev0);
  if (ctx->ev1) cudaEventDestroy(ctx->ev1);
  for (int i = 0; i < TF_GPU_MAX_FRAMES; i++)
    if (ctx->ev_f32[i]) cudaEventDestroy(ctx->ev_f32[i]);
  if (ctx->ev_s16) cudaEventDestroy(ctx->ev_s16);
  if (ctx->stream2) {
    cudaStreamSynchronize(ctx->stream2);
    cudaStreamDestroy(ctx->stream2);
  }
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

const char *tf_gpu_last_error(const tf_gpu_ctx *ctx) { return ctx ? ctx->err : "no context (no CUDA device?)"; }

int tf_gpu_cache_frame(tf_gpu_ctx *ctx, const tf_gpu_frame *frame) {
  if (!ctx || !frame) return TF_GPU_ERR_INVALID;
  if (!frame->frame_id) return fail(ctx, TF_GPU_ERR_INVALID, "frame_id 0 cannot be cached");
  CU(cudaSetDevice(ctx->device));
  CallScope scope(ctx);
  DevFrame *d;
  const int num_planes = frame->plane[1] ? 3 : 1;
  int rc = get_frame(ctx, frame, num_planes, &d);
  if (rc) return rc;
  CU(cudaStreamSynchronize(ctx->copy_stream));
  return TF_GPU_OK;
}

int tf_gpu_cache_frame_async(tf_gpu_ctx *ctx, const tf_gpu_frame *frame) {
  if (!ctx || !frame) return TF_GPU_ERR_INVALID;
  if (!frame->frame_id) return fail(ctx, TF_GPU_ERR_INVALID, "frame_id 0 cannot be cached");
  CU(cudaSetDevice(ctx->device));
  if (ctx->async_upload_pending) {  // at most one asynchronous upload outstanding (see tf_gpu.h)
    CU(cudaEventSynchronize(ctx->ev_async_upload));
    ctx->async_upload_pending = false;
  }
  CallScope scope(ctx);
  DevFrame *d;
  const int num_planes = frame->plane[1] ? 3 : 1;
  int rc = get_frame(ctx, frame, num_planes, &d);
  if (rc) return rc;
  CU(cudaEventRecord(ctx->ev_async_upload, ctx->copy_stream));
  ctx->async_upload_pending = true;
  return TF_GPU_OK;
}

int tf_gpu_cache_frame_device(tf_gpu_ctx *ctx, const tf_gpu_frame *frame, void *stream) {
  if (!ctx || !frame) return TF_GPU_ERR_INVALID;
  ctx->last_launches = 0;
  if (!frame->frame_id) return fail(ctx, TF_GPU_ERR_INVALID, "frame_id 0 cannot be cached");
  const int num_planes = frame->plane[1] ? 3 : 1;
  Geometry g;
  if (!make_geometry(frame, num_planes, &g)) return fail(ctx, TF_GPU_ERR_INVALID, "bad frame geometry");
  CU(cudaSetDevice(ctx->device));
  // Everything the ingest kernels will read is checked here, before anything is enqueued: a plane is device (or
  // managed) memory of this context's device, and its crop area, rows `stride` samples apart, lies inside the
  // allocation the pointer belongs to (or in allocations mapped contiguously after it).
  const size_t es = g.is_hbd ? 2 : 1;
  for (int p = 0; p < num_planes; p++) {
    const int k = p > 0;
    if (!frame->plane[p]) return fail(ctx, TF_GPU_ERR_INVALID, "frame plane %d is NULL", p);
    if (g.crop_w[k] <= 0 || g.crop_h[k] <= 0 || g.aligned_w[k] < g.crop_w[k] || g.aligned_h[k] < g.crop_h[k])
      return fail(ctx, TF_GPU_ERR_INVALID, "plane %d: bad crop / aligned size", p);
    if (frame->stride[k] < g.crop_w[k])
      return fail(ctx, TF_GPU_ERR_INVALID, "plane %d: stride %d is smaller than the crop width %d", p, frame->stride[k], g.crop_w[k]);
    char what[16];
    snprintf(what, sizeof(what), "plane %d", p);
    const int rc = check_device_extent(ctx, frame->plane[p], ((size_t)(g.crop_h[k] - 1) * frame->stride[k] + g.crop_w[k]) * es,
                                       es, what);
    if (rc) return rc;
  }
  CallScope scope(ctx);
  FrameSource src;
  src.device = true;
  src.stream = (cudaStream_t)stream;
  DevFrame *d;
  int rc = get_frame(ctx, frame, num_planes, &d, src);
  if (rc) return rc;
  // the producer may overwrite or free the planes in its stream order (a resident frame: its last load)
  CU(cudaStreamWaitEvent(src.stream, d->ready, 0));
  return TF_GPU_OK;
}

int tf_gpu_device_border(void) { return DEV_BORDER; }

int tf_gpu_debug_read_plane(tf_gpu_ctx *ctx, uint64_t frame_id, int plane, void *dst, int dst_stride, int x0, int y0,
                            int w, int h) {
  if (!ctx || !dst || plane < 0 || plane > TF_GPU_DEBUG_ROWSUM_PLANE || w <= 0 || h <= 0) return TF_GPU_ERR_INVALID;
  CU(cudaSetDevice(ctx->device));
  DevFrame *d = find_cached(ctx, frame_id, nullptr);
  if (!d) return fail(ctx, TF_GPU_ERR_INVALID, "frame id %llu is not resident", (unsigned long long)frame_id);
  const Geometry &g = d->g;
  const bool rowsum = plane == TF_GPU_DEBUG_ROWSUM_PLANE;
  if (!rowsum && plane >= g.num_planes) return fail(ctx, TF_GPU_ERR_INVALID, "plane not present");
  const int k = !rowsum && plane > 0;
  const size_t es = (rowsum || g.is_hbd) ? 2 : 1;
  if (x0 < -g.bx[k] || y0 < -g.by[k] || x0 + w > g.pitch[k] - g.bx[k] || y0 + h > g.rows[k] - g.by[k])
    return fail(ctx, TF_GPU_ERR_INVALID, "rectangle outside the device allocation");
  CU(cudaStreamSynchronize(ctx->copy_stream));
  const void *p00 = rowsum ? (const void *)d->rs00 : d->p00[plane];
  const char *src = (const char *)p00 + ((long long)y0 * g.pitch[k] + x0) * (long long)es;
  CU(cudaMemcpy2D(dst, (size_t)dst_stride * es, src, (size_t)g.pitch[k] * es, (size_t)w * es, h, cudaMemcpyDeviceToHost));
  return TF_GPU_OK;
}

int tf_gpu_evict_frame(tf_gpu_ctx *ctx, uint64_t frame_id) {
  if (!ctx) return TF_GPU_ERR_INVALID;
  for (auto &d : ctx->cache)
    if (d.valid && d.frame_id == frame_id) d.valid = false;
  return TF_GPU_OK;
}

int tf_gpu_estimate_noise(tf_gpu_ctx *ctx, const tf_gpu_frame *frame, int plane, int bit_depth, int edge_thresh,
                          double *noise_level) {
  if (!ctx || !frame || !noise_level) return TF_GPU_ERR_INVALID;
  if (plane < 0 || plane > 2) return fail(ctx, TF_GPU_ERR_INVALID, "plane out of range");
  if (bit_depth != 8 && bit_depth != 10 && bit_depth != 12) return fail(ctx, TF_GPU_ERR_INVALID, "bit_depth must be 8, 10 or 12");
  if (!frame->is_hbd && bit_depth != 8) return fail(ctx, TF_GPU_ERR_INVALID, "8-bit container needs bit_depth 8");
  CU(cudaSetDevice(ctx->device));
  CallScope scope(ctx);
  ctx->last_launches = 0;
  cudaStream_t ns = ctx->noise_stream;  // not the main stream: a window submitted earlier keeps running
  DevFrame *d;
  const int num_planes = frame->plane[1] ? 3 : 1;
  if (plane >= num_planes) return fail(ctx, TF_GPU_ERR_INVALID, "plane not present");
  int rc = get_frame(ctx, frame, num_planes, &d);
  if (rc) return rc;
  CU(cudaStreamWaitEvent(ns, d->ready, 0));
  const Geometry &g = d->g;
  const int k = plane > 0;
  const int w = g.crop_w[k], h = g.crop_h[k];
  CU(cudaMemsetAsync(ctx->d_noise, 0, 2 * sizeof(unsigned long long), ns));
  if (w > 2 && h > 2) {
    const long long n = (long long)(w - 2) * (h - 2);
    const int threads = 256;
    long long blocks = (n + threads - 1) / threads;
    if (blocks > ctx->num_sms * 8) blocks = ctx->num_sms * 8;
    if (g.is_hbd)
      noise_kernel<uint16_t><<<(int)blocks, threads, 0, ns>>>((const uint16_t *)d->p00[plane], g.pitch[k], w, h, bit_depth, edge_thresh, ctx->d_noise);
    else
      noise_kernel<uint8_t><<<(int)blocks, threads, 0, ns>>>((const uint8_t *)d->p00[plane], g.pitch[k], w, h, bit_depth, edge_thresh, ctx->d_noise);
    CU(cudaGetLastError());
    ctx->last_launches++;
  }
  CU(cudaMemcpyAsync(ctx->h_noise, ctx->d_noise, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ns));
  CU(cudaStreamSynchronize(ns));
  const long long accum = (long long)ctx->h_noise[0];
  const int count = (int)ctx->h_noise[1];
  // temporal_filter.c:1193, SQRT_PI_BY_2 :1148
  *noise_level = (count < 16) ? -1.0 : (double)accum / (6 * count) * 1.25331413732;
  return TF_GPU_OK;
}

int tf_gpu_submit(tf_gpu_ctx *ctx, const tf_gpu_params *params, const tf_gpu_frame *frames, tf_gpu_frame *out,
                  int64_t diff_sum_sse[2], uint64_t *ticket) {
  if (!ticket) return TF_GPU_ERR_INVALID;
  return submit_impl(ctx, params, frames, out, diff_sum_sse, nullptr, ticket);
}

int tf_gpu_wait(tf_gpu_ctx *ctx, uint64_t ticket) {
  if (!ctx) return TF_GPU_ERR_INVALID;
  Ticket &t = ctx->tickets[ticket % 8];
  if (!t.pending || t.id != ticket) return fail(ctx, TF_GPU_ERR_INVALID, "unknown ticket");
  CU(cudaSetDevice(ctx->device));
  CU(cudaEventSynchronize(t.ev));
  t.pending = false;
  if (t.want_diff) {
    t.diff_dst[0] = (int64_t)ctx->h_diff[2 * (ticket % 8)];
    t.diff_dst[1] = (int64_t)ctx->h_diff[2 * (ticket % 8) + 1];
  }
  float ms = 0.f;
  if (cudaEventElapsedTime(&ms, t.te.ev0, t.te.ev1) == cudaSuccess) ctx->last_kernel_ms = ms;
  ctx->last_ev = &t.te;
  return TF_GPU_OK;
}

int tf_gpu_filter_dump(tf_gpu_ctx *ctx, const tf_gpu_params *params, const tf_gpu_frame *frames, tf_gpu_frame *out,
                       int64_t diff_sum_sse[2], const tf_gpu_dump *dump) {
  uint64_t t;
  int rc = submit_impl(ctx, params, frames, out, diff_sum_sse, dump, &t);
  if (rc) return rc;
  return tf_gpu_wait(ctx, t);
}

int tf_gpu_filter(tf_gpu_ctx *ctx, const tf_gpu_params *params, const tf_gpu_frame *frames, tf_gpu_frame *out,
                  int64_t diff_sum_sse[2]) {
  return tf_gpu_filter_dump(ctx, params, frames, out, diff_sum_sse, nullptr);
}

int tf_gpu_filter_resident_async(tf_gpu_ctx *ctx, const tf_gpu_params *params, const uint64_t *frame_ids) {
  if (!ctx || !frame_ids) return TF_GPU_ERR_INVALID;
  int rc = validate_params(ctx, params);
  if (rc) return rc;
  CU(cudaSetDevice(ctx->device));
  CallScope scope(ctx);
  ctx->last_launches = 0;
  DevFrame *devf[TF_GPU_MAX_FRAMES];
  for (int i = 0; i < params->num_frames; i++) {
    devf[i] = find_cached(ctx, frame_ids[i], nullptr);
    if (!devf[i]) return fail(ctx, TF_GPU_ERR_INVALID, "frame id %llu is not resident", (unsigned long long)frame_ids[i]);
    if (!(devf[i]->g == devf[0]->g)) return fail(ctx, TF_GPU_ERR_INVALID, "frames of one window must share geometry");
    devf[i]->last_use = ++ctx->use_counter;
    devf[i]->pinned_epoch = ctx->epoch;
  }
  const Geometry &g = devf[0]->g;
  rc = validate_geometry(ctx, params, g);
  if (rc) return rc;
  rc = alloc_dev_frame(ctx, &ctx->out, g);
  if (rc) return rc;
  // slot 8 of the FRAME_DIFF ring belongs to the resident path (slots 0..7: tickets)
  unsigned long long *d_diff = ctx->d_diff + 2 * 8;
  CU(cudaMemsetAsync(d_diff, 0, 2 * sizeof(unsigned long long), ctx->stream));
  rc = launch_filter(ctx, params, devf, g, d_diff, nullptr, &ctx->res_ev);
  if (rc) return rc;
  CU(cudaMemcpyAsync(ctx->h_diff + 2 * 8, d_diff, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
  return TF_GPU_OK;
}

int tf_gpu_filter_resident_result(tf_gpu_ctx *ctx, int64_t diff_sum_sse[2], float *time_ms) {
  if (!ctx) return TF_GPU_ERR_INVALID;
  CU(cudaSetDevice(ctx->device));
  CU(cudaStreamSynchronize(ctx->stream));
  if (diff_sum_sse) {
    diff_sum_sse[0] = (int64_t)ctx->h_diff[2 * 8];
    diff_sum_sse[1] = (int64_t)ctx->h_diff[2 * 8 + 1];
  }
  float ms = 0.f;
  CU(cudaEventElapsedTime(&ms, ctx->res_ev.ev0, ctx->res_ev.ev1));
  ctx->last_ev = &ctx->res_ev;
  ctx->last_kernel_ms = ms;
  if (time_ms) *time_ms = ms;
  return TF_GPU_OK;
}

int tf_gpu_filter_resident(tf_gpu_ctx *ctx, const tf_gpu_params *params, const uint64_t *frame_ids,
                           int64_t diff_sum_sse[2], float *time_ms) {
  const int rc = tf_gpu_filter_resident_async(ctx, params, frame_ids);
  if (rc) return rc;
  return tf_gpu_filter_resident_result(ctx, diff_sum_sse, time_ms);
}

int tf_gpu_filter_batch_async(tf_gpu_ctx *ctx, int n, const tf_gpu_params *params, const uint64_t *const *frame_ids) {
  static_assert(MAXB == TF_GPU_MAX_BATCH, "device batch size and ABI batch size must agree");
  if (!ctx) return TF_GPU_ERR_INVALID;
  // every check comes before anything is enqueued or pinned: a rejected batch leaves the context as it was
  if (n < 1 || n > TF_GPU_MAX_BATCH) return fail(ctx, TF_GPU_ERR_INVALID, "batch of %d windows out of [1,%d]", n, TF_GPU_MAX_BATCH);
  if (!params || !frame_ids) return fail(ctx, TF_GPU_ERR_INVALID, "params / frame_ids is NULL");
  for (int w = 0; w < n; w++) {
    const tf_gpu_params *p = &params[w];
    if (!frame_ids[w]) return fail(ctx, TF_GPU_ERR_INVALID, "frame_ids[%d] is NULL", w);
    int rc = validate_params(ctx, p);
    if (rc) return rc;
    if (p->out_row_end > p->out_row_begin)
      return fail(ctx, TF_GPU_ERR_INVALID, "window %d: a batch filters whole frames (no out_row_begin / out_row_end)", w);
    if (p->extend_output_borders)
      return fail(ctx, TF_GPU_ERR_INVALID, "window %d: a batch does not extend output borders", w);
  }
  if (ctx->peer_out[0] || ctx->peer_out[1] || ctx->peer_out[2])
    return fail(ctx, TF_GPU_ERR_INVALID, "an output plane is imported from another rank: a batch writes only its own outputs");
  if (ctx->collect_counters) return fail(ctx, TF_GPU_ERR_INVALID, "work counters are not collected for batches");
  {
    uint64_t ids[TF_GPU_MAX_BATCH * TF_GPU_MAX_FRAMES];
    int nd = 0;
    for (int w = 0; w < n; w++)
      for (int i = 0; i < params[w].num_frames; i++) {
        int j = 0;
        while (j < nd && ids[j] != frame_ids[w][i]) j++;
        if (j == nd) ids[nd++] = frame_ids[w][i];
      }
    if (nd > (int)ctx->cache.size())
      return fail(ctx, TF_GPU_ERR_INVALID, "the batch reads %d distinct frames, the frame cache holds %d", nd, (int)ctx->cache.size());
  }
  CU(cudaSetDevice(ctx->device));
  DevFrame *devf[TF_GPU_MAX_BATCH][TF_GPU_MAX_FRAMES];
  for (int w = 0; w < n; w++)
    for (int i = 0; i < params[w].num_frames; i++) {
      devf[w][i] = find_cached(ctx, frame_ids[w][i], nullptr);
      if (!devf[w][i])
        return fail(ctx, TF_GPU_ERR_INVALID, "window %d: frame id %llu is not resident", w, (unsigned long long)frame_ids[w][i]);
      if (!(devf[w][i]->g == devf[0][0]->g)) return fail(ctx, TF_GPU_ERR_INVALID, "window %d: the frames of a batch must share one geometry", w);
    }
  const Geometry &g = devf[0][0]->g;
  for (int w = 0; w < n; w++) {
    const int rc = validate_geometry(ctx, &params[w], g);
    if (rc) return rc;
  }
  CallScope scope(ctx);
  ctx->last_launches = 0;
  ctx->batch_n = 0;
  for (int w = 0; w < n; w++)
    for (int i = 0; i < params[w].num_frames; i++) {
      DevFrame *d = devf[w][i];
      if (d->pinned_epoch != ctx->epoch) CU(cudaStreamWaitEvent(ctx->stream, d->ready, 0));
      d->last_use = ++ctx->use_counter;
      d->pinned_epoch = ctx->epoch;
    }
  for (int w = 0; w < n; w++) {
    const int rc = alloc_dev_frame(ctx, &ctx->bout[w], g);
    if (rc) return rc;
  }
  if (!ctx->d_bdiff) CU(cudaMalloc(&ctx->d_bdiff, TF_GPU_MAX_BATCH * 2 * sizeof(unsigned long long)));
  if (!ctx->h_bdiff) CU(cudaMallocHost(&ctx->h_bdiff, TF_GPU_MAX_BATCH * 2 * sizeof(unsigned long long)));
  const int rc = launch_filter_batch(ctx, n, params, devf, g, &ctx->batch_ev);
  if (rc) return rc;
  CU(cudaMemcpyAsync(ctx->h_bdiff, ctx->d_bdiff, (size_t)n * 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
  for (int w = 0; w < n; w++) ctx->batch_planes[w] = params[w].num_planes;
  ctx->batch_n = n;
  return TF_GPU_OK;
}

int tf_gpu_filter_batch_result(tf_gpu_ctx *ctx, int64_t (*diff_sum_sse)[2], float *time_ms) {
  if (!ctx) return TF_GPU_ERR_INVALID;
  if (!ctx->batch_n) return fail(ctx, TF_GPU_ERR_INVALID, "no batch has been enqueued");
  CU(cudaSetDevice(ctx->device));
  CU(cudaStreamSynchronize(ctx->stream));
  if (diff_sum_sse)
    for (int w = 0; w < ctx->batch_n; w++) {
      diff_sum_sse[w][0] = (int64_t)ctx->h_bdiff[2 * w];
      diff_sum_sse[w][1] = (int64_t)ctx->h_bdiff[2 * w + 1];
    }
  float ms = 0.f;
  CU(cudaEventElapsedTime(&ms, ctx->batch_ev.ev0, ctx->batch_ev.ev1));
  ctx->last_ev = &ctx->batch_ev;
  ctx->last_kernel_ms = ms;
  if (time_ms) *time_ms = ms;
  return TF_GPU_OK;
}

int tf_gpu_download_batch_output(tf_gpu_ctx *ctx, int window, tf_gpu_frame *out) {
  if (!ctx || !out) return TF_GPU_ERR_INVALID;
  if (window < 0 || window >= ctx->batch_n) return fail(ctx, TF_GPU_ERR_INVALID, "window %d is not in the last batch (%d windows)", window, ctx->batch_n);
  CU(cudaSetDevice(ctx->device));
  const DevFrame &d = ctx->bout[window];
  int rc = download_rows(ctx, d, out, 0, (d.g.crop_h[0] + 31) / 32, ctx->stream, ctx->batch_planes[window]);
  if (rc) return rc;
  CU(cudaStreamSynchronize(ctx->stream));
  return TF_GPU_OK;
}

int tf_gpu_batch_output_device_plane(tf_gpu_ctx *ctx, int window, int plane, void **dptr, size_t *pitch_bytes,
                                     int *rows, int *row_bytes) {
  if (!ctx || plane < 0 || plane > 2) return TF_GPU_ERR_INVALID;
  if (window < 0 || window >= ctx->batch_n) return fail(ctx, TF_GPU_ERR_INVALID, "window %d is not in the last batch (%d windows)", window, ctx->batch_n);
  if (plane >= ctx->batch_planes[window] || !ctx->bout[window].p00[plane])
    return fail(ctx, TF_GPU_ERR_INVALID, "window %d filters %d plane(s): no plane %d", window, ctx->batch_planes[window], plane);
  device_plane(ctx->bout[window], plane, dptr, pitch_bytes, rows, row_bytes);
  return TF_GPU_OK;
}

int tf_gpu_download_output(tf_gpu_ctx *ctx, tf_gpu_frame *out, int row_begin, int row_end) {
  if (!ctx || !out) return TF_GPU_ERR_INVALID;
  if (!ctx->out.base[0]) return fail(ctx, TF_GPU_ERR_INVALID, "no output on the device yet");
  CU(cudaSetDevice(ctx->device));
  const int mb_rows = (ctx->out.g.crop_h[0] + 31) / 32;
  if (row_end <= row_begin) {
    row_begin = 0;
    row_end = mb_rows;
  }
  if (row_begin < 0) row_begin = 0;
  if (row_end > mb_rows) row_end = mb_rows;
  int rc = download_rows(ctx, ctx->out, out, row_begin, row_end, ctx->stream);
  if (rc) return rc;
  CU(cudaStreamSynchronize(ctx->stream));
  return TF_GPU_OK;
}

int tf_gpu_output_device_plane(tf_gpu_ctx *ctx, int plane, void **dptr, size_t *pitch_bytes, int *rows,
                               int *row_bytes) {
  if (!ctx || plane < 0 || plane > 2 || !ctx->out.p00[plane]) return TF_GPU_ERR_INVALID;
  device_plane(ctx->out, plane, dptr, pitch_bytes, rows, row_bytes);
  return TF_GPU_OK;
}

int tf_gpu_output_ipc_export(tf_gpu_ctx *ctx, int plane, unsigned char handle[TF_GPU_IPC_HANDLE_BYTES], size_t *offset_bytes,
                             size_t *pitch_bytes) {
  if (!ctx || !handle || plane < 0 || plane > 2) return TF_GPU_ERR_INVALID;
  if (!ctx->out.base[plane]) return fail(ctx, TF_GPU_ERR_INVALID, "no output plane %d on the device yet", plane);
  static_assert(sizeof(cudaIpcMemHandle_t) == TF_GPU_IPC_HANDLE_BYTES, "handle size");
  CU(cudaSetDevice(ctx->device));
  cudaIpcMemHandle_t h;
  CU(cudaIpcGetMemHandle(&h, ctx->out.base[plane]));
  memcpy(handle, &h, sizeof(h));
  if (offset_bytes) *offset_bytes = (size_t)((char *)ctx->out.p00[plane] - (char *)ctx->out.base[plane]);
  if (pitch_bytes) *pitch_bytes = (size_t)ctx->out.g.pitch[plane > 0] * (ctx->out.g.is_hbd ? 2 : 1);
  return TF_GPU_OK;
}

int tf_gpu_output_ipc_import(tf_gpu_ctx *ctx, int plane, const unsigned char *handle, size_t offset_bytes, size_t pitch_bytes) {
  if (!ctx || plane < 0 || plane > 2) return TF_GPU_ERR_INVALID;
  CU(cudaSetDevice(ctx->device));
  CU(cudaStreamSynchronize(ctx->stream));  // no kernel may still be writing through the old mapping
  if (ctx->peer_base[plane]) {
    CU(cudaIpcCloseMemHandle(ctx->peer_base[plane]));
    ctx->peer_base[plane] = ctx->peer_out[plane] = nullptr;
    ctx->peer_pitch[plane] = 0;
  }
  if (!handle) return TF_GPU_OK;
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof(h));
  void *base = nullptr;
  CU(cudaIpcOpenMemHandle(&base, h, cudaIpcMemLazyEnablePeerAccess));
  ctx->peer_base[plane] = base;
  ctx->peer_out[plane] = (char *)base + offset_bytes;
  ctx->peer_pitch[plane] = pitch_bytes;
  return TF_GPU_OK;
}

namespace {

// The params of a batched search: the caller's search fields, and window fields that validate_params accepts --
// frame 0 the source, frames 1 .. num_frames - 1 the references, luma only.
tf_gpu_params search_params(const tf_gpu_params &in, int num_frames) {
  tf_gpu_params p = in;
  p.num_frames = num_frames;
  p.filter_frame_idx = 0;
  p.num_planes = 1;
  return p;
}

// A batched search item's position against the rule tf_motion_batch_kernel applies to items in device memory.
int check_item_position(tf_gpu_ctx *ctx, const tf_gpu_params &p, int i, int x, int y) {
  if (!item_position_ok(x, y, p.mi_rows, p.mi_cols))
    return fail(ctx, TF_GPU_ERR_INVALID, "item %d: block position (%d, %d) not supported", i, x, y);
  return TF_GPU_OK;
}

// The checks the motion-search and predictor entry points make before anything is enqueued or pinned, short of the
// items (the synchronous search reads them on the host, the device calls leave them to the kernel) and of where the
// item and output buffers live.  src_id: the search's source, NULL for the predictor, whose frames are the
// references alone.  num_planes: the planes the call reads (the search: 1).  n == 0 passes without the frame checks:
// the caller returns TF_GPU_OK.  Otherwise *p holds the call's params and devf[0 ..] the slots in frame order (the
// source first, then the references).
int check_resident_call(tf_gpu_ctx *ctx, const tf_gpu_params *params, const uint64_t *src_id, const uint64_t *ref_ids,
                        int num_refs, int block_size, int n, int num_planes, tf_gpu_params *p, DevFrame **devf) {
  if (!params || !ref_ids) return fail(ctx, TF_GPU_ERR_INVALID, "NULL argument");
  if (block_size != 16 && block_size != 32) return fail(ctx, TF_GPU_ERR_INVALID, "block_size must be 16 or 32");
  if (n < 0) return fail(ctx, TF_GPU_ERR_INVALID, "negative item count");
  if (num_refs < 1 || num_refs > TF_GPU_MAX_FRAMES - 1)
    return fail(ctx, TF_GPU_ERR_INVALID, "num_refs %d out of [1,%d]", num_refs, TF_GPU_MAX_FRAMES - 1);
  if (n == 0) return TF_GPU_OK;
  const int nsrc = src_id ? 1 : 0;
  *p = search_params(*params, nsrc + num_refs);
  p->num_planes = num_planes;
  int rc = validate_params(ctx, p);
  if (rc) return rc;
  for (int f = 0; f < nsrc + num_refs; f++) {
    const uint64_t id = f < nsrc ? *src_id : ref_ids[f - nsrc];
    devf[f] = find_cached(ctx, id, nullptr);
    if (!devf[f]) return fail(ctx, TF_GPU_ERR_INVALID, "frame id %llu is not resident", (unsigned long long)id);
    if (!(devf[f]->g == devf[0]->g)) return fail(ctx, TF_GPU_ERR_INVALID, "the source and references must share one geometry");
  }
  return validate_geometry(ctx, p, devf[0]->g);
}

// One caller buffer of a stream-ordered call: `bytes` from `ptr`, `align`-byte aligned.
struct DeviceSpan {
  const void *ptr;
  size_t bytes, align;
  const char *what;
};
// Each buffer is device or managed memory of the context's device with its extent inside its allocation
// (check_device_extent), and no two overlap.
int check_device_spans(tf_gpu_ctx *ctx, const DeviceSpan *s, int count) {
  for (int i = 0; i < count; i++) {
    const int rc = check_device_extent(ctx, s[i].ptr, s[i].bytes, s[i].align, s[i].what);
    if (rc) return rc;
  }
  for (int i = 0; i < count; i++)
    for (int j = i + 1; j < count; j++) {
      const uintptr_t a = (uintptr_t)s[i].ptr, b = (uintptr_t)s[j].ptr;
      if (a < b + s[j].bytes && b < a + s[i].bytes) return fail(ctx, TF_GPU_ERR_INVALID, "%s and %s overlap", s[i].what, s[j].what);
    }
  return TF_GPU_OK;
}

// Pins the slots for the current epoch (so that done_ev covers the kernels that read them, for a later eviction)
// and makes the main stream wait for each slot's upload or ingest.
int pin_slots(tf_gpu_ctx *ctx, DevFrame *const *devf, int count) {
  for (int f = 0; f < count; f++) {
    DevFrame *d = devf[f];
    if (d->pinned_epoch != ctx->epoch) CU(cudaStreamWaitEvent(ctx->stream, d->ready, 0));
    d->last_use = ++ctx->use_counter;
    d->pinned_epoch = ctx->epoch;
  }
  return TF_GPU_OK;
}

// The body of a stream-ordered call: `enqueue` runs on the main stream after the work already on the caller's
// `stream`, and `stream` waits for it, so that done_ev covers the call's kernel (see get_frame) and the caller may
// consume the outputs in its own stream order.  Never blocks the host.
extern "C++" template <class F>
int on_caller_stream(tf_gpu_ctx *ctx, void *stream, F &&enqueue) {
  const cudaStream_t s = (cudaStream_t)stream;
  CU(cudaEventRecord(ctx->ev_search_src, s));
  CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_search_src, 0));
  const int rc = enqueue();
  if (rc) return rc;
  CU(cudaEventRecord(ctx->ev_search_done, ctx->stream));
  CU(cudaStreamWaitEvent(s, ctx->ev_search_done, 0));
  return TF_GPU_OK;
}

// The search itself, on the main stream, for both entry points: pins the slots, and makes one launch over
// items / results in device memory; `timed`: ctx->ev0 / ev1 around the launch.
int enqueue_motion_search(tf_gpu_ctx *ctx, const tf_gpu_params &p, DevFrame *const *devf, int num_refs, int block_size,
                          const MotionItem *d_items, MotionResult *d_res, int n, bool timed) {
  const int rc = pin_slots(ctx, devf, 1 + num_refs);
  if (rc) return rc;
  const Geometry &g = devf[0]->g;
  KParams K;
  fill_kparams(ctx, &p, g, K);
  // frames past the references are the source's: an item's ref is checked in the kernel, and even a wrong check
  // could then not reach a null or stale frame pointer
  for (int f = 0; f < MAXF; f++) K.frm[f][0] = devf[f <= num_refs ? f : 0]->p00[0];
  if (timed) CU(cudaEventRecord(ctx->ev0, ctx->stream));
  if (g.is_hbd) {
    if (block_size == 32) tf_motion_batch_kernel<uint16_t, 32><<<n, 32, SearchSmem<uint16_t, 32>::TOTAL, ctx->stream>>>(K, d_items, d_res, n);
    else tf_motion_batch_kernel<uint16_t, 16><<<n, 32, SearchSmem<uint16_t, 16>::TOTAL, ctx->stream>>>(K, d_items, d_res, n);
  } else {
    if (block_size == 32) tf_motion_batch_kernel<uint8_t, 32><<<n, 32, SearchSmem<uint8_t, 32>::TOTAL, ctx->stream>>>(K, d_items, d_res, n);
    else tf_motion_batch_kernel<uint8_t, 16><<<n, 32, SearchSmem<uint8_t, 16>::TOTAL, ctx->stream>>>(K, d_items, d_res, n);
  }
  CU(cudaGetLastError());
  ctx->last_launches++;
  if (timed) CU(cudaEventRecord(ctx->ev1, ctx->stream));
  return TF_GPU_OK;
}

}  // namespace

int tf_gpu_fullpel_search_batch(tf_gpu_ctx *ctx, const tf_gpu_params *params, const tf_gpu_frame *src,
                                const tf_gpu_frame *ref, int block_size, const tf_gpu_search_item *items, int n,
                                tf_gpu_search_result *results) {
  if (!ctx) return TF_GPU_ERR_INVALID;
  if (!params || !src || !ref || !items || !results) return fail(ctx, TF_GPU_ERR_INVALID, "NULL argument");
  if (block_size != 16 && block_size != 32) return fail(ctx, TF_GPU_ERR_INVALID, "block_size must be 16 or 32");
  if (n < 0) return fail(ctx, TF_GPU_ERR_INVALID, "negative item count");
  if (n == 0) return TF_GPU_OK;
  static_assert(sizeof(tf_gpu_search_item) == sizeof(SearchItem) && sizeof(tf_gpu_search_result) == sizeof(SearchResult),
                "ABI structs and device structs must agree");
  tf_gpu_params p = search_params(*params, 2);  // only the search fields are read
  if (p.subpel_iters_per_step < 1) p.subpel_iters_per_step = 1;
  int rc = validate_params(ctx, &p);
  if (rc) return rc;
  CU(cudaSetDevice(ctx->device));
  CallScope scope(ctx);
  ctx->last_launches = 0;
  DevFrame *ds = nullptr, *dr = nullptr;
  rc = get_frame(ctx, src, src->plane[1] ? 3 : 1, &ds);
  if (rc) return rc;
  rc = get_frame(ctx, ref, ref->plane[1] ? 3 : 1, &dr);
  if (rc) return rc;
  if (!(ds->g == dr->g)) return fail(ctx, TF_GPU_ERR_INVALID, "src and ref must share geometry");
  const Geometry &g = ds->g;
  rc = validate_geometry(ctx, &p, g);
  if (rc) return rc;
  for (int i = 0; i < n; i++) {
    rc = check_item_position(ctx, p, i, items[i].x, items[i].y);
    if (rc) return rc;
  }
  KParams K;
  fill_kparams(ctx, &p, g, K);
  rc = ensure_dump(ctx, 10, (size_t)n * sizeof(SearchItem));
  if (rc) return rc;
  rc = ensure_dump(ctx, 11, (size_t)n * sizeof(SearchResult));
  if (rc) return rc;
  SearchItem *d_items = (SearchItem *)ctx->d_dump[10];
  SearchResult *d_res = (SearchResult *)ctx->d_dump[11];
  CU(cudaMemcpyAsync(d_items, items, (size_t)n * sizeof(SearchItem), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaStreamWaitEvent(ctx->stream, ds->ready, 0));
  CU(cudaStreamWaitEvent(ctx->stream, dr->ready, 0));
  if (g.is_hbd) {
    const uint16_t *a = (const uint16_t *)ds->p00[0], *b = (const uint16_t *)dr->p00[0];
    if (block_size == 32) tf_fullpel_batch_kernel<uint16_t, 32><<<n, 32, SearchSmem<uint16_t, 32>::TOTAL, ctx->stream>>>(K, a, b, d_items, d_res, n);
    else tf_fullpel_batch_kernel<uint16_t, 16><<<n, 32, SearchSmem<uint16_t, 16>::TOTAL, ctx->stream>>>(K, a, b, d_items, d_res, n);
  } else {
    const uint8_t *a = (const uint8_t *)ds->p00[0], *b = (const uint8_t *)dr->p00[0];
    if (block_size == 32) tf_fullpel_batch_kernel<uint8_t, 32><<<n, 32, SearchSmem<uint8_t, 32>::TOTAL, ctx->stream>>>(K, a, b, d_items, d_res, n);
    else tf_fullpel_batch_kernel<uint8_t, 16><<<n, 32, SearchSmem<uint8_t, 16>::TOTAL, ctx->stream>>>(K, a, b, d_items, d_res, n);
  }
  CU(cudaGetLastError());
  ctx->last_launches++;
  CU(cudaMemcpyAsync(results, d_res, (size_t)n * sizeof(SearchResult), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return TF_GPU_OK;
}

int tf_gpu_motion_search_batch(tf_gpu_ctx *ctx, const tf_gpu_params *params, uint64_t src_id, const uint64_t *ref_ids,
                               int num_refs, int block_size, const tf_gpu_motion_item *items, int n,
                               tf_gpu_motion_result *results) {
  static_assert(sizeof(tf_gpu_motion_item) == sizeof(MotionItem) && sizeof(tf_gpu_motion_result) == sizeof(MotionResult),
                "ABI structs and device structs must agree");
  if (!ctx) return TF_GPU_ERR_INVALID;
  // every check comes before anything is enqueued or pinned: a rejected call leaves the context as it was
  if (!items || !results) return fail(ctx, TF_GPU_ERR_INVALID, "NULL argument");
  tf_gpu_params p;
  DevFrame *devf[TF_GPU_MAX_FRAMES];
  int rc = check_resident_call(ctx, params, &src_id, ref_ids, num_refs, block_size, n, 1, &p, devf);
  if (rc || n == 0) return rc;
  for (int i = 0; i < n; i++) {
    rc = check_item_position(ctx, p, i, items[i].x, items[i].y);
    if (rc) return rc;
    if (items[i].ref < 0 || items[i].ref >= num_refs)
      return fail(ctx, TF_GPU_ERR_INVALID, "item %d: ref %d out of [0,%d)", i, (int)items[i].ref, num_refs);
  }
  CU(cudaSetDevice(ctx->device));
  CallScope scope(ctx);
  ctx->last_launches = 0;
  rc = ensure_dump(ctx, 12, (size_t)n * sizeof(MotionItem));
  if (rc) return rc;
  rc = ensure_dump(ctx, 13, (size_t)n * sizeof(MotionResult));
  if (rc) return rc;
  MotionItem *d_items = (MotionItem *)ctx->d_dump[12];
  MotionResult *d_res = (MotionResult *)ctx->d_dump[13];
  CU(cudaMemcpyAsync(d_items, items, (size_t)n * sizeof(MotionItem), cudaMemcpyHostToDevice, ctx->stream));
  rc = enqueue_motion_search(ctx, p, devf, num_refs, block_size, d_items, d_res, n, true);
  if (rc) return rc;
  CU(cudaMemcpyAsync(results, d_res, (size_t)n * sizeof(MotionResult), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  float ms = 0.f;
  CU(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
  ctx->last_kernel_ms = ms;
  return TF_GPU_OK;
}

int tf_gpu_motion_search_device(tf_gpu_ctx *ctx, const tf_gpu_params *params, uint64_t src_id, const uint64_t *ref_ids,
                                int num_refs, int block_size, const tf_gpu_motion_item *items, int n,
                                tf_gpu_motion_result *results, void *stream) {
  static_assert(TF_GPU_MOTION_REJECTED == MOTION_REJECTED, "header and kernel must agree on the rejection sentinel");
  if (!ctx) return TF_GPU_ERR_INVALID;
  // every check comes before anything is enqueued or pinned: a rejected call leaves the context as it was
  if (!items || !results) return fail(ctx, TF_GPU_ERR_INVALID, "NULL argument");
  tf_gpu_params p;
  DevFrame *devf[TF_GPU_MAX_FRAMES];
  int rc = check_resident_call(ctx, params, &src_id, ref_ids, num_refs, block_size, n, 1, &p, devf);
  if (rc || n == 0) return rc;
  CU(cudaSetDevice(ctx->device));
  const size_t bytes = (size_t)n * sizeof(MotionItem);
  const DeviceSpan spans[2] = { { items, bytes, 4, "items" }, { results, bytes, 4, "results" } };
  rc = check_device_spans(ctx, spans, 2);
  if (rc) return rc;
  CallScope scope(ctx);
  ctx->last_launches = 0;
  ctx->last_kernel_ms = 0.f;  // not timed: the call does not wait for the kernel
  return on_caller_stream(ctx, stream, [&]() -> int {
    return enqueue_motion_search(ctx, p, devf, num_refs, block_size, (const MotionItem *)items, (MotionResult *)results,
                                 n, false);
  });
}

// Far MVs (tf_predict_kernel): the origin clamp is exact when every plane's border covers a sub-block's 12-tap
// footprint plus the load margins: b >= w + 11 + PRED_ML + PRED_MR, w <= 16 >> ss, b = DEV_BORDER >> ss.
static_assert(DEV_BORDER >= 16 + 11 + PRED_ML + PRED_MR && (DEV_BORDER >> 1) >= 8 + 11 + PRED_ML + PRED_MR,
              "the device border must hold a far-MV predictor footprint");

int tf_gpu_predict_device(tf_gpu_ctx *ctx, const tf_gpu_params *params, const uint64_t *ref_ids, int num_refs,
                          int block_size, const tf_gpu_predict_item *items, int n, void *pred, int32_t *status,
                          void *stream) {
  static_assert(sizeof(tf_gpu_predict_item) == sizeof(tf_gpu_motion_item) &&
                    offsetof(tf_gpu_predict_item, row) == offsetof(tf_gpu_motion_item, start_row) &&
                    offsetof(tf_gpu_predict_item, col) == offsetof(tf_gpu_motion_item, start_col) &&
                    offsetof(tf_gpu_predict_item, ref) == offsetof(tf_gpu_motion_item, ref),
                "a predictor item has the layout of a motion-search item");
  static_assert(sizeof(tf_gpu_predict_item) == sizeof(PredictItem), "ABI struct and device struct must agree");
  if (!ctx) return TF_GPU_ERR_INVALID;
  // every check comes before anything is enqueued or pinned: a rejected call leaves the context as it was
  if (!items || !pred || !status) return fail(ctx, TF_GPU_ERR_INVALID, "NULL argument");
  tf_gpu_params p;
  DevFrame *devf[TF_GPU_MAX_FRAMES];
  int rc = check_resident_call(ctx, params, nullptr, ref_ids, num_refs, block_size, n, params ? params->num_planes : 0,
                               &p, devf);
  if (rc || n == 0) return rc;
  CU(cudaSetDevice(ctx->device));
  const Geometry &g = devf[0]->g;
  const size_t es = g.is_hbd ? 2 : 1;
  const int num_pels =
      block_size * block_size + (p.num_planes > 1 ? 2 * (block_size >> g.ss_x) * (block_size >> g.ss_y) : 0);
  const DeviceSpan spans[3] = { { items, (size_t)n * sizeof(PredictItem), 4, "items" },
                                { pred, (size_t)n * num_pels * es, es, "pred" },
                                { status, (size_t)n * sizeof(int32_t), 4, "status" } };
  rc = check_device_spans(ctx, spans, 3);
  if (rc) return rc;
  CallScope scope(ctx);
  ctx->last_launches = 0;
  ctx->last_kernel_ms = 0.f;  // not timed: the call does not wait for the kernel
  return on_caller_stream(ctx, stream, [&]() -> int {
    const int rc2 = pin_slots(ctx, devf, num_refs);
    if (rc2) return rc2;
    KParams K;
    fill_kparams(ctx, &p, g, K);
    K.num_pels = num_pels;
    // frames past the references are the first reference's: a wrong ref check could not reach a null pointer
    for (int f = 0; f < MAXF; f++)
      for (int pl = 0; pl < p.num_planes; pl++) K.frm[f][pl] = devf[f < num_refs ? f : 0]->p00[pl];
    const long long grid = block_size == 32 ? n : ((long long)n + FILT_WARPS - 1) / FILT_WARPS;
    const PredictItem *d_items = (const PredictItem *)items;
    if (g.is_hbd)
      tf_predict_kernel<uint16_t><<<(unsigned)grid, FILT_THREADS, 0, ctx->stream>>>(
          K, d_items, (uint16_t *)pred, status, n, block_size, g.bx[1], g.by[1], g.bx[0]);
    else
      tf_predict_kernel<uint8_t><<<(unsigned)grid, FILT_THREADS, 0, ctx->stream>>>(
          K, d_items, (uint8_t *)pred, status, n, block_size, g.bx[1], g.by[1], g.bx[0]);
    CU(cudaGetLastError());
    ctx->last_launches++;
    return TF_GPU_OK;
  });
}

int tf_gpu_host_register(tf_gpu_ctx *ctx, void *ptr, size_t bytes) {
  if (!ctx || !ptr) return TF_GPU_ERR_INVALID;
  CU(cudaSetDevice(ctx->device));
  CU(cudaHostRegister(ptr, bytes, cudaHostRegisterDefault));
  return TF_GPU_OK;
}

int tf_gpu_host_unregister(tf_gpu_ctx *ctx, void *ptr) {
  if (!ctx || !ptr) return TF_GPU_ERR_INVALID;
  CU(cudaSetDevice(ctx->device));
  CU(cudaHostUnregister(ptr));
  return TF_GPU_OK;
}

int tf_gpu_collect_counters(tf_gpu_ctx *ctx, int enable) {
  if (!ctx) return TF_GPU_ERR_INVALID;
  ctx->collect_counters = enable != 0;
  return TF_GPU_OK;
}

int tf_gpu_read_counters(tf_gpu_ctx *ctx, uint64_t counters[4]) {
  if (!ctx || !counters) return TF_GPU_ERR_INVALID;
  CU(cudaSetDevice(ctx->device));
  CU(cudaStreamSynchronize(ctx->stream));
  CU(cudaMemcpy(ctx->h_ctr, ctx->d_ctr, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  for (int i = 0; i < 4; i++) counters[i] = ctx->h_ctr[i];
  return TF_GPU_OK;
}

int tf_gpu_last_kernel_times(tf_gpu_ctx *ctx, float ms[3]) {
  if (!ctx || !ms) return TF_GPU_ERR_INVALID;
  ms[0] = ms[1] = ms[2] = 0.f;
  if (!ctx->split_valid || !ctx->last_ev) return TF_GPU_OK;
  const CallEvents &te = *ctx->last_ev;
  CU(cudaSetDevice(ctx->device));
  CU(cudaEventSynchronize(te.ev1));
  CU(cudaEventElapsedTime(&ms[0], te.ev0, te.evk[0]));
  CU(cudaEventElapsedTime(&ms[1], te.evk[0], te.evk[1]));
  CU(cudaEventElapsedTime(&ms[2], te.evk[1], te.ev1));
  return TF_GPU_OK;
}

int tf_gpu_last_stats(const tf_gpu_ctx *ctx, int *kernel_launches, float *filter_kernel_ms) {
  if (!ctx) return TF_GPU_ERR_INVALID;
  if (kernel_launches) *kernel_launches = ctx->last_launches;
  if (filter_kernel_ms) *filter_kernel_ms = ctx->last_kernel_ms;
  return TF_GPU_OK;
}

int tf_gpu_event_record(tf_gpu_ctx *ctx, int slot) {
  if (!ctx || slot < 0 || slot > 3) return TF_GPU_ERR_INVALID;
  CU(cudaSetDevice(ctx->device));
  CU(cudaEventRecord(ctx->user_ev[slot], ctx->stream));
  return TF_GPU_OK;
}

int tf_gpu_event_elapsed_ms(tf_gpu_ctx *ctx, int slot_begin, int slot_end, float *ms) {
  if (!ctx || !ms || slot_begin < 0 || slot_begin > 3 || slot_end < 0 || slot_end > 3) return TF_GPU_ERR_INVALID;
  CU(cudaSetDevice(ctx->device));
  CU(cudaEventSynchronize(ctx->user_ev[slot_end]));
  CU(cudaEventElapsedTime(ms, ctx->user_ev[slot_begin], ctx->user_ev[slot_end]));
  return TF_GPU_OK;
}

int tf_gpu_synchronize(tf_gpu_ctx *ctx) {
  if (!ctx) return TF_GPU_ERR_INVALID;
  CU(cudaSetDevice(ctx->device));
  CU(cudaStreamSynchronize(ctx->stream));
  CU(cudaStreamSynchronize(ctx->out_stream));
  CU(cudaStreamSynchronize(ctx->copy_stream));
  CU(cudaStreamSynchronize(ctx->noise_stream));
  ctx->async_upload_pending = false;
  return TF_GPU_OK;
}

int tf_gpu_microbench(tf_gpu_ctx *ctx, int kind, double *giga_lane_ops_per_s) {
  if (!ctx || !giga_lane_ops_per_s || kind < 0 || kind > 5) return TF_GPU_ERR_INVALID;
  CU(cudaSetDevice(ctx->device));
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, ctx->device));
  unsigned *d_out = nullptr;
  CU(cudaMalloc(&d_out, 4));
  const int blocks = prop.multiProcessorCount * 4, threads = 256, iters = kind == 5 ? 2000 : 4000;
  float best = 1e30f;
  for (int rep = 0; rep < 4; rep++) {
    CU(cudaEventRecord(ctx->ev0, ctx->stream));
    switch (kind) {
      case 0: microbench_kernel<0><<<blocks, threads, 0, ctx->stream>>>(d_out, iters, 12345u + rep); break;
      case 1: microbench_kernel<1><<<blocks, threads, 0, ctx->stream>>>(d_out, iters, 12345u + rep); break;
      case 2: microbench_kernel<2><<<blocks, threads, 0, ctx->stream>>>(d_out, iters, 12345u + rep); break;
      case 3: microbench_kernel<3><<<blocks, threads, 0, ctx->stream>>>(d_out, iters, 12345u + rep); break;
      case 4: microbench_kernel<4><<<blocks, threads, 0, ctx->stream>>>(d_out, iters, 12345u + rep); break;
      default: microbench_kernel<5><<<blocks, threads, 0, ctx->stream>>>(d_out, iters, 12345u + rep); break;
    }
    CU(cudaEventRecord(ctx->ev1, ctx->stream));
    CU(cudaEventSynchronize(ctx->ev1));
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    if (rep > 0 && ms < best) best = ms;
  }
  cudaFree(d_out);
  const double lane_ops = (double)blocks * threads * (double)iters * 64.0;
  *giga_lane_ops_per_s = lane_ops / (best * 1e-3) / 1e9;
  return TF_GPU_OK;
}

}  // extern "C"
