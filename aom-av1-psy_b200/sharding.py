"""Work partitioning across the GPUs of one box (SURVEY 8e); one process per GPU.

Two independent axes, no exchange during compute:
  * window-parallel: one ARF window per rank (round robin) -- no collective;
  * slab-parallel (4K): the block rows of ONE window are split into contiguous
    ranges; every rank needs all whole frames (the search range is +-1023 px, so
    a halo smaller than the frame cannot be bit-exact) and computes only its
    output rows (tf_gpu_params.out_row_begin/end), which are then gathered to
    rank 0 straight from the library's device output planes, plus a 16-byte
    all-reduce for FRAME_DIFF (integer sums: order independent); or, without any
    gather, every rank stores its rows straight into rank 0's planes over NVLink
    (CUDA IPC peer mapping, `connect_peer_output`).  When only one rank holds the window's frames,
    `replicate_frames` broadcasts them over NVLink and every rank ingests them from device memory.
The reference's counterpart is the row job queue of av1/encoder/ethread.c:2062-2189
(workers share tf_ctx->output_frame and add their FRAME_DIFF under a mutex, :2161-2173).

`SlabWindow` is the slab driver used by bench.py and the multi-GPU tests; the collective
calls go through the `dist` module handed in (torch.distributed: NCCL on GPUs, gloo in
the CPU tests), so the same code runs in both.
"""


def slab_rows(mb_rows, world, rank):
    """Contiguous block-row range [begin, end) of `rank` out of `world`."""
    return (mb_rows * rank) // world, (mb_rows * (rank + 1)) // world


def max_slab_rows(mb_rows, world):
    return max(slab_rows(mb_rows, world, r)[1] - slab_rows(mb_rows, world, r)[0] for r in range(world))


def window_owner(window_index, world):
    """Round-robin owner of an independent window."""
    return window_index % world


def merge_slabs(slabs, mb_rows, world, block_h):
    """Stack per-rank row slabs (each padded to max_slab_rows*block_h rows) into the full plane."""
    import numpy as np
    rows = []
    for r, s in enumerate(slabs):
        b, e = slab_rows(mb_rows, world, r)
        rows.append(s[: (e - b) * block_h])
    return np.concatenate(rows, axis=0)


class SlabWindow:
    """One window filtered by `world` ranks, each computing the block rows slab_rows(mb_rows, world, rank)."""

    def __init__(self, mb_rows, world, rank, ss_y=1, num_planes=3):
        self.mb_rows, self.world, self.rank = mb_rows, world, rank
        self.begin, self.end = slab_rows(mb_rows, world, rank)
        self.pad_rows = max_slab_rows(mb_rows, world)
        self.block_h = [32] + [32 >> ss_y] * (num_planes - 1)
        self._recv = None
        self._stage, self._stage_meta = None, None  # replicate_frames' staging tensors and what they were made for

    def params(self, p):
        """The window's parameters restricted to this rank's rows."""
        return dict(p, out_row_begin=self.begin, out_row_end=self.end)

    # ---- device side: zero-copy views of the library's output planes -------------------------
    def device_slabs(self, ctx, torch, device):
        """This rank's slab of every output plane as a flat uint8 tensor of pad_rows block rows (whole
        pitched rows; the device border below the frame absorbs the padding of the shorter slabs)."""
        out = []
        for pl, bh in enumerate(self.block_h):
            ptr, pitch, rows, row_bytes = ctx.output_device_plane(pl)

            class _View:  # __cuda_array_interface__ holder
                pass
            v = _View()
            v.__cuda_array_interface__ = {"shape": ((self.mb_rows + 1) * bh * pitch,), "typestr": "|u1",
                                          "data": (ptr, False), "version": 3}
            t = torch.as_tensor(v, device=device)
            lo = self.begin * bh * pitch
            out.append(t[lo:lo + self.pad_rows * bh * pitch])
        return out

    def device_planes(self, ctx, torch, device):
        """The library's whole output planes (all block rows, whole pitched rows) as flat uint8 tensors."""
        out = []
        for pl, bh in enumerate(self.block_h):
            ptr, pitch, rows, row_bytes = ctx.output_device_plane(pl)

            class _View:
                pass
            v = _View()
            v.__cuda_array_interface__ = {"shape": (self.mb_rows * bh * pitch,), "typestr": "|u1",
                                          "data": (ptr, False), "version": 3}
            out.append(torch.as_tensor(v, device=device))
        return out

    # ---- peer-store variant: no gather, every rank writes its rows into the owner's planes over NVLink -------
    def connect_peer_output(self, ctx, dist, owner=0):
        """The owner exports its device output planes (CUDA IPC), every other rank imports them: from now on a
        rank's filter call stores its block rows straight into the owner's frame (tf_gpu_output_ipc_*).  The
        owner's planes must exist (one filter call of this geometry has run on every rank)."""
        box, err = [None], None
        if self.rank == owner:
            try:
                box = [[ctx.output_ipc_export(pl) for pl in range(len(self.block_h))]]
            except Exception as e:  # the broadcast below still has to happen on every rank
                err = e
        dist.broadcast_object_list(box, src=owner)
        if err is not None:
            raise err
        if box[0] is None:
            raise RuntimeError("the owner rank could not export its output planes")
        if self.rank != owner:
            for pl, (handle, off, pitch) in enumerate(box[0]):
                ctx.output_ipc_import(pl, handle, off, pitch)

    def disconnect_peer_output(self, ctx, owner=0):
        if self.rank != owner:
            for pl in range(len(self.block_h)):
                ctx.output_ipc_import(pl, None)

    def finish_peer(self, diff, dist):
        """After this rank's filter call has completed: sum FRAME_DIFF over the ranks; past this all-reduce every
        rank's rows are in the owner's planes."""
        dist.all_reduce(diff)
        return diff

    # ---- frame replication: the window's pixels cross PCIe once per box ---------------------------------------
    def replicate_frames(self, ctx, dist, torch, frames, ids, owner=0, device=None):
        """Put the window's frames into every rank's frame cache when only `owner` holds them.  frames / ids:
        on the owner, per frame (y, u, v) (u, v None for monochrome) as host arrays or CUDA tensors, and the frame
        ids; ignored elsewhere.  The owner stages each plane in a device tensor, dist.broadcast sends it to every
        rank's staging tensor (shapes, dtypes and ids go first with broadcast_object_list, so the other ranks need
        no pixels), and every rank, owner included, ingests it with ctx.cache_frame_tensor.  The staging tensors
        are reused by the next window of the same geometry.  device: where staging lives (default: the current
        CUDA device under NCCL, the CPU otherwise).  Returns the ids."""
        if device is None:
            device = (torch.device("cuda", torch.cuda.current_device()) if dist.get_backend() == "nccl"
                      else torch.device("cpu"))
        def as_tensor(a):  # collectives carry 16-bit samples as int16 (the ingest takes int16 and uint16 alike)
            if not isinstance(a, torch.Tensor):
                return torch.from_numpy(a.view("int16") if a.dtype.itemsize == 2 else a)
            return a.view(torch.int16) if a.dtype == getattr(torch, "uint16", None) else a

        src = []
        box = [None]
        if self.rank == owner:
            src = [[as_tensor(a) for a in planes if a is not None] for planes in frames]
            box = [([int(i) for i in ids], [[(tuple(t.shape), str(t.dtype)) for t in ts] for ts in src])]
        dist.broadcast_object_list(box, src=owner)
        out_ids, meta = box[0]
        if self._stage is None or self._stage_meta != (meta, device):
            # byte tensors on the wire (NCCL and gloo have no 16-bit integer type), sample-typed views for the ingest
            self._stage = []
            for planes in meta:
                views = []
                for (h, w), dt in planes:
                    dt = getattr(torch, dt.split(".")[-1])
                    views.append(torch.empty((h, w * dt.itemsize), dtype=torch.uint8, device=device).view(dt))
                self._stage.append(views)
            self._stage_meta = (meta, device)
        for f, planes in enumerate(self._stage):
            for p, t in enumerate(planes):
                if self.rank == owner:
                    t.copy_(src[f][p])
                dist.broadcast(t.view(torch.uint8), src=owner)
            ctx.cache_frame_tensor(out_ids[f], *planes)
        return out_ids

    # ---- collective ---------------------------------------------------------------------------
    def gather(self, slabs, diff, dist, torch):
        """slabs: this rank's per-plane tensors (any dtype / device, equal shapes across ranks); diff: this
        rank's FRAME_DIFF [sum, sse] (int64 tensor on the same device).  Returns (per-plane list of the
        `world` slabs on rank 0 else None, the summed FRAME_DIFF on every rank)."""
        if self._recv is None or any(r is not None and r[0].shape != s.shape for r, s in zip(self._recv, slabs)):
            self._recv = [[torch.empty_like(s) for _ in range(self.world)] if self.rank == 0 else None for s in slabs]
        for s, r in zip(slabs, self._recv):
            dist.gather(s, r, dst=0)
        dist.all_reduce(diff)
        return self._recv if self.rank == 0 else None, diff

    def assemble(self, gathered, pitch_elems, cat):
        """Rank 0: the full planes [mb_rows * block_h, pitch] from the gathered slabs; `cat` joins a list of
        row blocks (torch.cat / numpy.concatenate)."""
        planes = []
        for pl, bh in enumerate(self.block_h):
            parts = []
            for r, s in enumerate(gathered[pl]):
                b, e = slab_rows(self.mb_rows, self.world, r)
                parts.append(s.reshape(-1, pitch_elems[pl])[: (e - b) * bh])
            planes.append(cat(parts))
        return planes
