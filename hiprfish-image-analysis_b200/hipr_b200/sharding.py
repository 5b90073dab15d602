"""Multi-GPU host logic: one process per GPU (torch.distributed).

* Independent fields of view (BASELINE config 3) shard by index with NO data-path collective:
  rank r takes FOVs r, r + world, ...  (`fov_shard`).
* One stitched mosaic split across GPUs (config 5) is cut into row slabs.  The stencil runs on
  the 1-channel sum image, so the only exchange is a 5-row halo of that image with the slab
  above and below (`exchange_halo`, one batch of isend/irecv: NCCL send/recv over NVLink on
  GPUs), plus two tiny all-reduces: the global max/min of the sum image (`allreduce_range`) and,
  for per-cell spectra, the (L+1, C) partial sums and (L+1) integer pixel counts
  (`allreduce_cells`; integer counts stay exact).

The compute steps are the CUDA operators in hipr_b200.ops; `MosaicSlab` takes them as hooks so
the communication logic can be exercised on CPU tensors with the gloo backend in tests.
"""
import ctypes as C

import torch
import torch.distributed as dist

from . import tables
from ._lib import FLAVOURS, lib
from .ops import _call, _launch

HALO = 5   # (patch_size - 1) / 2 for the 11-sample lines every pipeline uses


def fov_shard(n_fov, rank, world):
    """Indices of the fields of view rank `rank` processes."""
    return list(range(rank, n_fov, world))


def slab_bounds(n_rows, rank, world):
    """Rows [r0, r1) of the mosaic owned by `rank`: contiguous, balanced, every rank >= HALO rows."""
    if n_rows < world * HALO:
        raise ValueError("mosaic of %d rows is too short for %d slabs" % (n_rows, world))
    base, extra = divmod(n_rows, world)
    r0 = rank * base + min(rank, extra)
    return r0, r0 + base + (1 if rank < extra else 0)


def exchange_halo(slab, group=None, halo=HALO):
    """slab (rows, W) -> (halo_top + rows + halo_bottom, W): rows from the neighbouring ranks above
    and below; the outer ranks get nothing on their outer side (the stencil clamps to the edge
    there, = np.pad(mode='edge')).  Returns (extended, n_top, n_bottom)."""
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    slab = slab.contiguous()
    up, down = rank - 1, rank + 1
    top = torch.empty((halo, slab.shape[1]), dtype=slab.dtype, device=slab.device) if up >= 0 else None
    bottom = torch.empty((halo, slab.shape[1]), dtype=slab.dtype, device=slab.device) if down < world else None
    ops = []
    peer = (lambda r: r) if group is None else (lambda r: dist.get_global_rank(group, r))
    send_up = slab[:halo].contiguous() if up >= 0 else None
    send_down = slab[-halo:].contiguous() if down < world else None
    if up >= 0:
        ops += [dist.P2POp(dist.isend, send_up, peer(up), group), dist.P2POp(dist.irecv, top, peer(up), group)]
    if down < world:
        ops += [dist.P2POp(dist.isend, send_down, peer(down), group),
                dist.P2POp(dist.irecv, bottom, peer(down), group)]
    if ops:
        for req in dist.batch_isend_irecv(ops):
            req.wait()
    parts = [p for p in (top, slab, bottom) if p is not None]
    return torch.cat(parts, dim=0), (halo if top is not None else 0), (halo if bottom is not None else 0)


def allreduce_range(vmax, vmin, group=None):
    """Global (max, min) from per-slab float64 scalars (1-element tensors)."""
    t = torch.stack([vmax.reshape(()), -vmin.reshape(())]).to(torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    return t[0:1].clone(), (-t[1:2]).clone()


def allreduce_cells(sums, counts, group=None, root=None):
    """Sum the per-slab (L+1, C) float64 channel sums and (L+1) int32 pixel counts in place: on every rank
    (root=None, all-reduce) or on rank `root` only (reduce: half the traffic; the other ranks' buffers are then
    partial sums and must not be used)."""
    if root is None:
        dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=group)
        dist.all_reduce(counts, op=dist.ReduceOp.SUM, group=group)
    else:
        dst = root if group is None else dist.get_global_rank(group, root)
        dist.reduce(sums, dst=dst, op=dist.ReduceOp.SUM, group=group)
        dist.reduce(counts, dst=dst, op=dist.ReduceOp.SUM, group=group)
    return sums, counts


class MosaicSlab:
    """One rank's row slab of a stitched mosaic: score map and per-cell spectra with the same
    results as the unsplit mosaic.

    hooks (defaults = the CUDA operators):
      channel_sum(cube_slab) -> (sum_slab float64 (rows, W), vmax (1,), vmin (1,))
      score(extended_sum, vmax, vmin, flavour) -> (rows_ext, W) score of the extended image
      accumulate(cube_slab, labels_slab, max_label) -> (sums, counts)
      finalize(sums, counts) -> (labels, area, avgint, avgint_norm)
    """

    def __init__(self, group=None, hooks=None):
        self.group = group
        self.hooks = hooks or _cuda_hooks()

    def score(self, cube_slab, flavour="F1"):
        s, vmax, vmin = self.hooks["channel_sum"](cube_slab)
        ext, n_top, n_bottom = exchange_halo(s, self.group)
        gmax, gmin = allreduce_range(vmax, vmin, self.group)
        full = self.hooks["score"](ext, gmax, gmin, flavour)
        return full[n_top: full.shape[0] - n_bottom]

    def cell_spectra(self, cube_slab, labels_slab, max_label, root=None):
        """The mosaic's cell table on every rank (root=None), or on rank `root` only (None elsewhere): the scripts
        write one table, and a reduce moves half the bytes of an all-reduce."""
        sums, counts = self.hooks["accumulate"](cube_slab, labels_slab, max_label)
        allreduce_cells(sums, counts, self.group, root)
        if root is not None and dist.get_rank(self.group) != root:
            return None
        return self.hooks["finalize"](sums, counts)


class P2PMosaicSlab:
    """MosaicSlab.score with the exchange done by this library's own kernels over NVLink peer memory instead of
    NCCL calls (csrc/mosaic_p2p.cu): the channel-sum kernel writes the slab's sums into a peer-mapped buffer, one
    push kernel stores the 5 edge rows into the neighbours' halo rows and the slab's max / min keys into every
    rank's table and releases a flag, one wait kernel acquires the flags and reduces the range.  torch.distributed
    is used once, at construction, to exchange the 64-byte IPC handles and the slab heights.

    One instance per (slab height, width); every rank must call score() the same number of times.

    Failure handling: if a peer does not deliver within `timeout_ms` (default ~10 s; a rank still loading its slab
    can be late by more: raise it), the wait kernel gives up instead of hanging the GPU and that call's score is
    overwritten with NaN on the device (hipr_mosaic_p2p_guard), so a stale halo never passes as a result;
    score(check=True) or check_peers() synchronises and raises instead.

    group: the process group used for the one-time handle exchange; a gloo group works (the data path never touches
    torch.distributed), which also lets two ranks share one GPU (cudaIpc mappings work within a device)."""

    def __init__(self, rows, width, group=None, timeout_ms=None):
        self.group = group
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        self.rows, self.width = int(rows), int(width)
        all_rows = [None] * self.world
        dist.all_gather_object(all_rows, self.rows, group=group)
        self.all_rows = [int(r) for r in all_rows]
        self.rows_max = max(self.all_rows)
        nbytes = lib().hipr_mosaic_p2p_bytes(self.rows_max, self.width, self.world)
        if nbytes <= 0:
            raise ValueError("mosaic geometry not supported by the peer-memory exchange")
        if timeout_ms is not None:
            _call("mosaic_p2p_set_timeout_ms", float(timeout_ms), what="p2p_set_timeout_ms")
        base = C.c_void_p()
        _call("p2p_alloc", C.byref(base), nbytes)
        self._own = base
        handle = (C.c_ubyte * 64)()
        _call("p2p_get_handle", base, handle)
        handles = [None] * self.world
        dist.all_gather_object(handles, bytes(handle), group=group)
        self._opened = []
        bases = []
        for r, h in enumerate(handles):
            if r == self.rank:
                bases.append(base.value)
                continue
            peer = C.c_void_p()
            buf = (C.c_ubyte * 64).from_buffer_copy(h)
            _call("p2p_open_handle", buf, C.byref(peer), what="p2p_open_handle (rank %d)" % r)
            self._opened.append(peer)
            bases.append(peer.value)
        self._bases = (C.c_void_p * self.world)(*bases)
        self.epoch = 0
        dev = torch.device("cuda", torch.cuda.current_device())
        self._keys = torch.empty(2, dtype=torch.int64, device=dev)
        self._range = torch.empty(2, dtype=torch.int64, device=dev)
        self._error = torch.zeros(1, dtype=torch.int32, device=dev)
        dist.barrier(group=group)        # every rank has opened every buffer before the first push

    def _rows_ptr(self, parity, with_top_halo):
        p = C.c_void_p()
        _call("mosaic_p2p_rows_ptr", self._own, self.rows_max, self.width, self.world, parity, int(with_top_halo),
              C.byref(p), what="p2p_rows_ptr")
        return p

    def score(self, cube_slab, flavour="F1", bands=0, check=False):
        """check=True: synchronise and raise if a peer timed out (otherwise a timed-out call returns NaN scores).
        bands >= 3 (F1 / F2): one call that also hides the stencil under the channel sum, band by band
        (hipr_mosaic_p2p_score; every tile quantised with its own range).  bands = 0: channel sum, exchange,
        stencil in order (bit-identical to MosaicSlab.score); F3 uses the exchanged global range."""
        if tuple(cube_slab.shape[:2]) != (self.rows, self.width) or cube_slab.dtype != torch.float32:
            raise ValueError("cube_slab must be (%d, %d, C) float32" % (self.rows, self.width))
        cube_slab = cube_slab.contiguous()
        Cn = cube_slab.shape[2]
        dev = cube_slab.device
        self.epoch += 1
        parity = self.epoch & 1
        rows_up = self.all_rows[self.rank - 1] if self.rank > 0 else 0
        if bands >= 3:
            tab = tables.line_table_2d(11, 9)
            out = torch.empty((self.rows, self.width), dtype=torch.float32, device=dev)
            _launch("mosaic_p2p_score", dev, cube_slab, Cn, self._bases, self.rank, self.world, self.rows, rows_up,
                    self.rows_max, self.width, parity, self.epoch, tab, FLAVOURS[flavour], int(bands), self._keys,
                    self._range, self._error, out)
            if check:
                self.check_peers()
            return out
        # channel sums straight into this rank's peer-mapped buffer (rows 5 .. 5 + rows of ext[parity])
        _launch("chansum", dev, cube_slab, None, self.rows * self.width, Cn, self._rows_ptr(parity, False), 1,
                self._keys, what="channel_sum")
        _launch("mosaic_p2p_exchange", dev, self._bases, self.rank, self.world, self.rows, rows_up, self.rows_max,
                self.width, parity, self._keys, self.epoch, self._range, self._error)
        n_top = HALO if self.rank > 0 else 0
        n_bottom = HALO if self.rank + 1 < self.world else 0
        Hs = self.rows + n_top + n_bottom
        tab = tables.line_table_2d(11, 9)
        out = torch.empty((Hs, self.width), dtype=torch.float32, device=dev)
        _launch("lne2d_q", dev, self._rows_ptr(parity, n_top > 0), Hs, self.width, self.width, 0, 1, 11, 9, tab,
                FLAVOURS[flavour], self._range if flavour not in ("F1", "F2") else None, out)
        _launch("mosaic_p2p_guard", dev, self._error, out, out.numel())
        if check:
            self.check_peers()
        return out[n_top: Hs - n_bottom]

    def check_peers(self):
        """Raises if a wait kernel timed out on a peer's flag (synchronises)."""
        if int(self._error.item()) != 0:
            raise RuntimeError("a peer did not deliver its halo rows in time")

    def close(self):
        torch.cuda.synchronize()
        dist.barrier(group=self.group)   # nobody still pushes into a buffer that is about to be freed
        for p in self._opened:
            lib().hipr_p2p_close_handle(p)
        self._opened = []
        if self._own is not None:
            lib().hipr_p2p_free(self._own)
            self._own = None


def _cuda_hooks():
    from . import ops

    def channel_sum(cube_slab):
        s, mk = ops.channel_sum(cube_slab, None, normalize=False, dtype=torch.float64, return_max=True)
        vmax, vmin = mk.values()
        return s, vmax, vmin

    def score(ext, gmax, gmin, flavour):
        # F1 / F2 are invariant to any affine map of the image: every 32x32 tile is quantised with its own
        # range (finer than the global one); F3's epsilon needs the global range
        keys = ops.MaxKey.from_values(gmax, gmin) if flavour not in ("F1", "F2") else None
        return ops.lne2d_fixed(ext, flavour, 11, 9, padded=False, range_keys=keys)

    return {"channel_sum": channel_sum, "score": score, "accumulate": ops.cell_spectra_accumulate,
            "finalize": ops.cell_spectra_finalize}
