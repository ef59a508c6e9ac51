"""Multi-GPU partitioning of the render path (SURVEY.md 8e): one process per GPU, torch.distributed for the
plumbing (NCCL on the GPUs, gloo in the CPU tests).

The reference has no counterpart (single thread, single GL context).  Two partitions exist, and neither puts a
collective on the data path of a render:

* viewpoint batch -- every viewpoint is an independent render against the same read-only DEM square, which each
  rank loads for itself.  Viewpoints are block-partitioned; outputs stay sharded on the rank that made them.
  Only reduced products (horizon profiles, a few bytes per image column) are gathered.  Viewsheds partition the same
  way; their per-vertex counts are summed over the ranks with one all_reduce (viewshed_counts_sharded).
* azimuth wedges  -- one giant panorama: rank g renders columns [edges[g], edges[g+1]), bit-identical to the same
  columns of an unsharded render.  PeerPanorama fuses the exchange into the renderer: each rank's resolve kernel
  stores its wedge straight into every rank's full panorama over NVLink (peer memory), a barrier is the only
  collective.  render_wedges() is the plain variant: private slabs + one all_gather + a strided placement.

Everything here except the two render_* drivers is device-agnostic tensor code, so the world_size-2 gloo tests
exercise exactly what runs over NCCL.
"""
import torch
import torch.distributed as dist


def block_partition(n, world, rank):
    """[lo, hi) of the items rank `rank` owns when n items are dealt out in contiguous, near-equal blocks."""
    if world <= 0 or not (0 <= rank < world):
        raise ValueError("bad rank %d of %d" % (rank, world))
    return n * rank // world, n * (rank + 1) // world


def wedge_edges(width, n_wedges):
    """Column edges of n_wedges near-equal azimuth wedges of a panorama `width` pixels wide."""
    if n_wedges <= 0 or n_wedges > width:
        raise ValueError("cannot cut %d columns into %d wedges" % (width, n_wedges))
    return [width * g // n_wedges for g in range(n_wedges + 1)]


def _world(group):
    if dist.is_available() and dist.is_initialized():
        return dist.get_world_size(group), dist.get_rank(group)
    return 1, 0


def stitch_wedges(slabs, edges):
    """slabs[g]: (H, >=w_g, ...) tensor whose first w_g = edges[g+1]-edges[g] columns are wedge g.  Returns the
    (H, W, ...) panorama."""
    first = slabs[0]
    W = edges[-1]
    out = first.new_empty((first.shape[0], W) + tuple(first.shape[2:]))
    for g, s in enumerate(slabs):
        x0, x1 = edges[g], edges[g + 1]
        out[:, x0:x1] = s[:, :x1 - x0]
    return out


def gather_wedges(local, edges, group=None):
    """All ranks contribute their wedge `local` (H, w_rank, ...); every rank gets the full (H, W, ...) panorama.
    Wedges may differ in width by one column; they travel padded to the widest one so that a single all_gather
    of equal-sized buffers does the exchange."""
    world, rank = _world(group)
    if world == 1:
        return stitch_wedges([local], edges)
    if len(edges) != world + 1:
        raise ValueError("need one wedge per rank: %d edges for %d ranks" % (len(edges), world))
    if local.shape[1] != edges[rank + 1] - edges[rank]:
        raise ValueError("rank %d holds %d columns, its wedge has %d" % (rank, local.shape[1], edges[rank + 1] - edges[rank]))
    wmax = max(edges[g + 1] - edges[g] for g in range(world))
    padded = local.new_zeros((local.shape[0], wmax) + tuple(local.shape[2:]))
    padded[:, :local.shape[1]] = local
    slabs = [torch.empty_like(padded) for _ in range(world)]
    dist.all_gather(slabs, padded.contiguous(), group=group)
    return stitch_wedges(slabs, edges)


def gather_blocks(local, n_total, group=None):
    """Inverse of block_partition for per-item results: `local` is (n_rank, ...) on every rank; returns
    (n_total, ...) on every rank.  Meant for reduced products, not for full images."""
    world, rank = _world(group)
    if world == 1:
        return local
    sizes = [block_partition(n_total, world, r) for r in range(world)]
    nmax = max(hi - lo for lo, hi in sizes)
    padded = local.new_zeros((nmax,) + tuple(local.shape[1:]))
    padded[:local.shape[0]] = local
    parts = [torch.empty_like(padded) for _ in range(world)]
    dist.all_gather(parts, padded.contiguous(), group=group)
    return torch.cat([p[:hi - lo] for p, (lo, hi) in zip(parts, sizes)], dim=0)


def horizon_profile(ranges):
    """Per image column: the row of the topmost terrain pixel (-1 if none) and the range there.
    ranges: (..., H, W) float tensor as render() returns it (top row first, < 0 where no terrain).
    Returns (rows int32 (..., W), range float32 (..., W)).  Device-agnostic reference implementation; the CUDA
    renderer has the same reduction as a kernel (horizonator_horizon_profile_device)."""
    hit = ranges > 0
    H = ranges.shape[-2]
    idx = torch.arange(H, device=ranges.device, dtype=torch.int32).view((1,) * (ranges.dim() - 2) + (H, 1))
    first = torch.where(hit, idx, torch.full_like(idx, H)).amin(dim=-2)
    rows = torch.where(first < H, first, torch.full_like(first, -1))
    rng = torch.gather(ranges, -2, first.clamp(max=H - 1).unsqueeze(-2).long()).squeeze(-2)
    rng = torch.where(first < H, rng, torch.full_like(rng, -1.0))
    return rows.to(torch.int32), rng.to(torch.float32)


# ---------------------------------------------------------------------------------------------- drivers (GPU)

def render_wedges(h, group=None, return_image=True, return_range=True):
    """One panorama of h's current view split by azimuth wedge over the ranks of `group`; every rank returns the
    full (H,W,3) uint8 / (H,W) float32 CUDA tensors.  All ranks must hold contexts of the same DEM, size and view."""
    world, rank = _world(group)
    W, H = h.width, h.height
    edges = wedge_edges(W, world)
    x0, x1 = edges[rank], edges[rank + 1]
    dev = torch.device("cuda", torch.cuda.current_device())
    img = torch.empty((H, x1 - x0, 3), dtype=torch.uint8, device=dev) if return_image else None
    rng = torch.empty((H, x1 - x0), dtype=torch.float32, device=dev) if return_range else None
    stream = torch.cuda.current_stream()
    h.render_wedge_device(x0, x1, img.data_ptr() if return_image else 0, rng.data_ptr() if return_range else 0,
                          stream.cuda_stream)
    out = []
    if return_image:
        out.append(gather_wedges(img, edges, group))
    if return_range:
        out.append(gather_wedges(rng, edges, group))
    return tuple(out)


class _DeviceArray:
    """Minimal __cuda_array_interface__ holder so that torch can view memory the library allocated."""

    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False), "version": 2}


class PeerPanorama:
    """One panorama split by azimuth wedge over the ranks and assembled WITHOUT a gather collective: every rank holds a
    full-size image and range buffer that its peers have mapped (CUDA IPC over NVLink/NVSwitch), and each rank's resolve
    kernel stores its wedge straight into all of them (horizonator_render_wedge_peers).  No collective library is
    involved in a render: the barriers that tell a rank its buffers are complete run on the GPUs through flags in peer
    memory (horizonator_peer_barrier), in stream order.

    Build once per context and size (collective: all ranks of `group` must construct it together), render() many
    times.  render() returns this rank's full (H,W,3) uint8 and (H,W) float32 tensors (views of the peer-mapped
    buffers: they are overwritten by the next render() of any rank)."""

    def __init__(self, h, group=None):
        self.h, self.group = h, group
        self.world, self.rank = _world(group)
        if self.world > 8:
            raise ValueError("at most 8 ranks (one NVSwitch domain) are supported")
        W, H = h.width, h.height
        self.W, self.H = W, H
        # column edges on multiples of 4 so that every wedge takes the vectorised resolve path
        self.edges = [((W * g // self.world) // 4) * 4 for g in range(self.world)] + [W]
        self.img_ptr, img_handle = h.peer_alloc(W * H * 3)
        self.rng_ptr, rng_handle = h.peer_alloc(W * H * 4)
        self.flag_ptr, flag_handle = h.peer_alloc(64)        # HORIZONATOR_PEER_FLAG_BYTES
        self.flags = torch.as_tensor(_DeviceArray(self.flag_ptr, (16,), "<u4"), device="cuda")
        self.flags.zero_()
        torch.cuda.synchronize()
        handles = [None] * self.world
        if self.world > 1:
            dist.all_gather_object(handles, (img_handle, rng_handle, flag_handle), group=group)   # also: flags are zeroed
        else:
            handles[0] = (img_handle, rng_handle, flag_handle)
        self.opened = []
        self.img_dst, self.rng_dst, self.flag_dst = [], [], []
        for r, (hi, hr, hf) in enumerate(handles):
            if r == self.rank:
                self.img_dst.append(self.img_ptr); self.rng_dst.append(self.rng_ptr); self.flag_dst.append(self.flag_ptr)
            else:
                pi, pr, pf = h.peer_open(hi), h.peer_open(hr), h.peer_open(hf)
                self.opened += [pi, pr, pf]
                self.img_dst.append(pi); self.rng_dst.append(pr); self.flag_dst.append(pf)
        self.epoch = 0
        self._timeouts_seen = 0
        self.image = torch.as_tensor(_DeviceArray(self.img_ptr, (H, W, 3), "|u1"), device="cuda")
        self.ranges = torch.as_tensor(_DeviceArray(self.rng_ptr, (H, W), "<f4"), device="cuda")
        if self.world > 1:
            dist.barrier(group=group)                        # everybody has mapped everything

    def render(self, root=None, strict=False):
        """Renders this rank's wedge of h's current view into everybody's buffers (root=None), or only into rank
        `root`'s (the others' buffers are then left as they were); all ranks call it together.

        The GPU-side barriers give up on a rank that does not arrive within their spin bound (a rank that died, or
        lags badly: first-call graph capture, host jitter) instead of hanging the GPU, and only count the time-out.
        The returned tensors are therefore complete only if timeouts() has not changed: strict=True checks that after
        waiting for the render (a host synchronisation per call) and raises RuntimeError if it has; callers that
        pipeline several renders should check timeouts() themselves once at the end."""
        before = self._timeouts_seen if strict else 0
        x0, x1 = self.edges[self.rank], self.edges[self.rank + 1]
        stream = torch.cuda.current_stream().cuda_stream
        img_dst = self.img_dst if root is None else [self.img_dst[root]]
        rng_dst = self.rng_dst if root is None else [self.rng_dst[root]]
        # both barriers run on the GPUs, in stream order: nothing here waits on the host
        self._barrier(stream)                       # nobody's stream is still reading the previous panorama
        self.h.render_wedge_peers(x0, x1, img_dst, rng_dst, stream)
        self._barrier(stream)                       # every wedge has landed everywhere
        if strict:
            now = self.timeouts()
            self._timeouts_seen = now
            if now != before:
                raise RuntimeError("PeerPanorama: %d GPU-side barrier(s) timed out; the panorama may be incomplete" % (now - before))
        return self.image, self.ranges

    def _barrier(self, stream):
        if self.world > 1:
            self.epoch += 1
            self.h.peer_barrier(self.rank, self.flag_dst, self.epoch, stream)

    def timeouts(self):
        """Number of GPU-side barriers of this rank that gave up waiting (0 unless a rank died or lagged badly)."""
        torch.cuda.synchronize()
        return int(self.flags[8].item())

    def close(self):
        torch.cuda.synchronize()
        for p in self.opened:
            self.h.peer_close(p)
        self.opened = []
        if self.world > 1:
            dist.barrier(group=self.group)          # peers have unmapped before the owner frees
        if self.img_ptr:
            self.image = self.ranges = self.flags = None
            self.h.peer_free(self.img_ptr); self.h.peer_free(self.rng_ptr); self.h.peer_free(self.flag_ptr)
            self.img_ptr = self.rng_ptr = self.flag_ptr = None


class HostPanorama:
    """One panorama split by azimuth wedge over the ranks and delivered to ONE host buffer -- where the reference's
    API puts its results (horizonator_render_offscreen) -- that all ranks share: a file in /dev/shm that every rank
    maps and page-locks, so that each rank's wedge travels over its own GPU's PCIe link (one GPU delivering the whole
    36000 x 4000 panorama moves 1 GB over a single link).  No collective on the data path; a barrier tells the ranks
    that the panorama is complete.  Build once per context and size (collective), render() many times; rank 0 owns the
    file.  `image` (H,W,3) uint8 and `ranges` (H,W) float32 are numpy views of the shared buffer."""

    def __init__(self, h, group=None, directory="/dev/shm"):
        import os
        import numpy as np
        from . import lib
        self.h, self.group, self._lib = h, group, lib
        self.world, self.rank = _world(group)
        W, H = h.width, h.height
        self.W, self.H = W, H
        # column edges on multiples of 4 so that every wedge takes the vectorised resolve path
        self.edges = [((W * g // self.world) // 4) * 4 for g in range(self.world)] + [W]
        name = [os.path.join(directory, "horizonator_pano_%d_%dx%d" % (os.getpid(), W, H))]
        nbytes = 7 * W * H
        if self.rank == 0:
            with open(name[0], "wb") as f:
                f.truncate(nbytes)
        if self.world > 1:
            dist.broadcast_object_list(name, src=0, group=group)      # also: the file exists
        self.path = name[0]
        self.buf = np.memmap(self.path, dtype=np.uint8, mode="r+", shape=(nbytes,))
        self.buf[::4096] = 0                                          # fault the pages in before they are locked
        self.registered = bool(lib.horizonator_host_register(self.buf.ctypes.data, nbytes))
        self.ranges = self.buf[:4 * W * H].view(np.float32).reshape(H, W)
        self.image = self.buf[4 * W * H:].reshape(H, W, 3)
        if self.world > 1:
            dist.barrier(group=group)

    def render(self):
        """Every rank renders its wedge of h's current view into the shared buffer; returns when all have."""
        self.h.render_wedge_host(self.edges[self.rank], self.edges[self.rank + 1], self.image, self.ranges)
        if self.world > 1:
            dist.barrier(group=self.group)
        return self.image, self.ranges

    def render_whole(self):
        """This rank alone renders all columns into the buffer (the one-GPU baseline)."""
        self.h.render_wedge_host(0, self.W, self.image, self.ranges)
        return self.image, self.ranges

    def close(self):
        import os
        if self.buf is not None:
            if self.registered:
                self._lib.horizonator_host_unregister(self.buf.ctypes.data)
            self.image = self.ranges = None
            self.buf = None
            if self.world > 1:
                dist.barrier(group=self.group)
            if self.rank == 0:
                try:
                    os.unlink(self.path)
                except OSError:
                    pass


def reduce_counts(counts, group=None, root=None):
    """Sums every rank's (N, N) viewshed counts: on every rank with root=None (all_reduce), else only on rank `root`
    (reduce; the other ranks' tensors then hold partial sums).  In place; returns `counts`."""
    world, _ = _world(group)
    if world > 1:
        if root is None:
            dist.all_reduce(counts, op=dist.ReduceOp.SUM, group=group)
        else:
            dist.reduce(counts, dst=root, op=dist.ReduceOp.SUM, group=group)
    return counts


def viewshed_counts_sharded(h, views, group=None, root=None, target_height=0.):
    """BASELINE configs[4] as a viewshed: block-partitions `views` over the ranks, adds this rank's viewsheds into
    counts on its own GPU (horizonator_viewshed_device) and sums the ranks' counts with one collective (see
    reduce_counts).  Returns the (N, N) int32 CUDA tensor: for every vertex of the loaded square, how many of the views
    see it.  All ranks must hold contexts of the same DEM square."""
    world, rank = _world(group)
    lo, hi = block_partition(len(views), world, rank)
    N = h.size
    counts = torch.zeros((N, N), dtype=torch.int32, device=torch.device("cuda", torch.cuda.current_device()))
    if hi > lo:
        h.viewshed_device(views[lo:hi], d_counts=counts.data_ptr(), target_height=target_height,
                          stream=torch.cuda.current_stream().cuda_stream)
    return reduce_counts(counts, group, root)


def render_batch_sharded(h, views, group=None, gather_profiles=True):
    """Block-partitions `views` over the ranks, renders this rank's share into device memory and returns
    (local_images, local_ranges, (lo, hi), profiles) -- profiles = (rows, range) of ALL views on every rank
    when gather_profiles, else None.  The full images never leave the GPU that rendered them."""
    world, rank = _world(group)
    lo, hi = block_partition(len(views), world, rank)
    W, H = h.width, h.height
    dev = torch.device("cuda", torch.cuda.current_device())
    img = torch.empty((hi - lo, H, W, 3), dtype=torch.uint8, device=dev)
    rng = torch.empty((hi - lo, H, W), dtype=torch.float32, device=dev)
    if hi > lo:
        h.render_batch_device(views[lo:hi], img.data_ptr(), rng.data_ptr(), torch.cuda.current_stream().cuda_stream)
    profiles = None
    if gather_profiles:
        rows, r = horizon_profile(rng)
        profiles = (gather_blocks(rows, len(views), group), gather_blocks(r, len(views), group))
    return img, rng, (lo, hi), profiles
