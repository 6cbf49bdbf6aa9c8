"""
Multi-GPU execution of the kernel-model path: one process per GPU, ``torch.distributed`` for the plumbing.

The reference parallelises over independent ``(band, block)`` units on a thread pool (fuse.py:396-408,
raster_pair.py:379-428); neighbouring blocks are only coupled through a fixed overlap of ``ceil(kernel / 2)`` proc-grid
pixels (utils.py:136-153).  Two regimes follow (SURVEY.md 8e):

* **Batch / mosaic** (`shard_sources`): independent source images are dealt round-robin to the ranks; the reference
  image is replicated.  No data-path collective at all.
* **One raster as row bands** (`RowBands`, `fuse_refspace_sharded`, `fit_apply_same_grid_sharded`): rank g owns a band
  of source rows whose edges coincide with proc-grid (reference) pixel rows.  Two things cross the interconnect:

  - **halo rows** (`exchange_halos`, `exchange_halos_inplace`): ``kh // 2`` proc-grid rows from each neighbour for the
    window sums (+ 2 for the up-sampler's taps when proc_crs = ref, 3 for lanczos; + 100 with R2 in-painting:
    `halo_rows`), sent point to point between row-band neighbours (NCCL P2P over NVLink on GPUs, gloo in the CPU
    tests).  Rows beyond the raster stay absent, which is the reference's zero padding (cv BORDER_CONSTANT).  proc_crs = ref exchanges rows of
    the DOWN-SAMPLED source (9 x 3000 float32 = 108 KB per neighbour and band for the 60k x 60k configuration); the
    same-grid path exchanges ``kh // 2`` rows of source and reference, received straight into the halo rows of
    pre-allocated planes (no copy of the band itself).
  - **block statistics** of gain-blk-offset (`block_norm_sharded`): ``_fit_block_norm`` (kernel_model.py:216-229) is a
    statistic of the WHOLE block, so its three streaming passes (counts + sums + 12-bit key histograms; squared
    deviations + next 12 bits; last 8 bits) run on each rank's own rows and every pass ends in one all-gather of the
    message (131 KB of accumulators, the shard's first / last valid pixels and its pairwise-leaf sums), merged in rank
    order by every rank: bit-identical statistics everywhere, and -- numpy's float32 pairwise ``np.std`` being replayed
    over the concatenation of the shards' valid pixels -- identical to the unsharded statistics.  No rank ever reads
    another rank's pixels beyond those few.

  Results equal the single-GPU results up to the summation order of the fit kernel's running sums (> 99.9 % of the
  parameters bit-identical; the block statistics are identical).

All timing of multi-GPU runs is done by the caller on the device (bench.py: CUDA events, max over ranks).
"""
from typing import List, NamedTuple, Optional, Sequence, Tuple

import torch
import torch.distributed as dist

from homonim_b200.geometry import Affine
from homonim_b200.raster_array import RasterArray


def _host_staged(t: torch.Tensor, group=None) -> bool:
    """ CUDA tensors over a back end without device support (gloo: several ranks sharing one GPU in the tests, or a box
    without NVLink / NCCL): the payload is staged through host memory.  NCCL moves device memory directly. """
    return t.is_cuda and dist.get_backend(group) != 'nccl'


def _run_p2p(sends, recvs, group=None) -> None:
    """ One batch of point-to-point transfers: ``sends`` / ``recvs`` are lists of ``(tensor view, peer)``; received rows
    land in the views. """
    if not sends and not recvs:
        return
    probe = (sends or recvs)[0][0]
    staged = _host_staged(probe, group)
    ops, landed = [], []
    for t, peer in sends:
        ops.append(dist.P2POp(dist.isend, t.cpu().contiguous() if staged else t, peer, group))
    for t, peer in recvs:
        buf = torch.empty(t.shape, dtype=t.dtype) if staged else t
        landed.append((t, buf))
        ops.append(dist.P2POp(dist.irecv, buf, peer, group))
    for req in dist.batch_isend_irecv(ops):
        req.wait()
    if staged:
        for t, buf in landed:
            t.copy_(buf)


_RANKS = {}


def _rank(group=None) -> int:
    """ ``dist.get_rank(group)``, cached per group (25 us per call otherwise, several calls per band and step). """
    key = id(group if group is not None else dist.group.WORLD)     # (a re-initialised default group is a new object)
    r = _RANKS.get(key)
    if r is None:
        r = _RANKS[key] = dist.get_rank(group)
    return r


def shard_sources(n_sources: int, rank: int, world_size: int) -> List[int]:
    """ Indexes of the independent source images this rank processes (round-robin; SURVEY.md 8e batch mode). """
    return list(range(rank, n_sources, world_size))


class RowBands(NamedTuple):
    """
    Partition of ``n_rows`` proc-grid rows into ``world_size`` contiguous bands, as even as possible.
    ``starts[g] .. starts[g + 1]`` is rank g's band (empty bands are allowed when there are more ranks than rows).
    """
    starts: Tuple[int, ...]

    @classmethod
    def split(cls, n_rows: int, world_size: int) -> 'RowBands':
        base, extra = divmod(int(n_rows), int(world_size))
        starts = [0]
        for g in range(world_size):
            starts.append(starts[-1] + base + (1 if g < extra else 0))
        return cls(tuple(starts))

    def band(self, rank: int) -> Tuple[int, int]:
        return self.starts[rank], self.starts[rank + 1]

    def size(self, rank: int) -> int:
        return self.starts[rank + 1] - self.starts[rank]

    def with_halo(self, rank: int, halo: int) -> Tuple[int, int]:
        """ Rank's band extended by ``halo`` rows on both sides, clipped to the raster. """
        a, b = self.band(rank)
        return max(a - halo, 0), min(b + halo, self.starts[-1])


def up_reach(upsampling) -> int:
    """ Parameter rows beyond a source row's cell that the up-sampler reads: 3 for lanczos' 6 taps, 2 for the 4-tap
    methods (cubic_spline, cubic, bilinear) -- and for nearest, which needs fewer. """
    from homonim_b200.enums import Resampling
    return 3 if Resampling.coerce(upsampling) == Resampling.lanczos else 2


def halo_rows(kernel_shape: Sequence[int], proc_crs_ref: bool, inpaint: bool, reach: int = 2) -> int:
    """
    Rows of proc-grid halo a row band needs on each side for its results to equal the whole-raster results:
    ``kh // 2`` for the window sums (the reference's block overlap uses the safe ``ceil(kh / 2)``, utils.py:136-153),
    + ``reach`` for the up-sampler's taps of the first / last up-sampled rows (proc_crs = ref; 2 for the 4-tap methods,
    3 for lanczos: `up_reach`), + 100 when in-painting is on (fillnodata's search radius, kernel_model.py:366).
    """
    return int(kernel_shape[0]) // 2 + (int(reach) if proc_crs_ref else 0) + (100 if inpaint else 0)


def _halo_peers(bands: RowBands, rank: int, halo: int) -> List[int]:
    """ Ranks that exchange rows with ``rank``: those whose band lies within ``halo`` rows of its band, on either side. """
    a, b = bands.band(rank)
    world = len(bands.starts) - 1
    peers = []
    for peer in range(rank - 1, -1, -1):                 # upwards until a band starts more than `halo` rows above
        peers.append(peer)
        if bands.starts[peer] <= a - halo:
            break
    for peer in range(rank + 1, world):                  # downwards likewise
        peers.append(peer)
        if bands.starts[peer + 1] >= b + halo:
            break
    return peers


def exchange_halos(local: torch.Tensor, bands: RowBands, halo: int, group=None) -> Tuple[torch.Tensor, int]:
    """
    Point-to-point halo exchange between row-band neighbours.

    ``local``: this rank's rows ``[..., n_local, width]`` of a raster split by ``bands``.  Returns ``(extended, top)``
    where ``extended`` holds the rows ``bands.with_halo(rank, halo)`` and ``top`` is the number of halo rows that were
    prepended.  A halo deeper than a neighbour's band is served by the next ranks as well.
    """
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    a, b = bands.band(rank)
    lo, hi = bands.with_halo(rank, halo)
    if world == 1 or halo == 0:
        return local, 0
    sends, recvs, recv_bufs = [], [], []
    lead = local.shape[:-2]
    width = local.shape[-1]
    for peer in _halo_peers(bands, rank, halo):
        pa, pb = bands.band(peer)
        plo, phi = bands.with_halo(peer, halo)
        # rows of mine that the peer needs
        s0, s1 = max(a, plo), min(b, phi)
        if s1 > s0:
            sends.append((local[..., s0 - a:s1 - a, :].contiguous(), peer))
        # rows of the peer that I need
        r0, r1 = max(pa, lo), min(pb, hi)
        if r1 > r0:
            buf = torch.empty(lead + (r1 - r0, width), dtype=local.dtype, device=local.device)
            recv_bufs.append((r0, buf))
            recvs.append((buf, peer))
    _run_p2p(sends, recvs, group)
    pieces = sorted(recv_bufs + [(a, local)], key=lambda t: t[0])
    extended = torch.cat([p for _, p in pieces], dim=-2) if len(pieces) > 1 else local
    return extended, a - lo


def all_gather_rows(local: torch.Tensor, bands: RowBands, group=None) -> torch.Tensor:
    """ All-gather row bands of unequal height into the whole ``[..., n_rows, width]`` plane on every rank. """
    world = dist.get_world_size(group)
    if world == 1:
        return local
    lead, width = local.shape[:-2], local.shape[-1]
    max_rows = max(bands.size(g) for g in range(world))
    padded = torch.zeros(lead + (max_rows, width), dtype=local.dtype, device=local.device)
    padded[..., :local.shape[-2], :] = local
    if _host_staged(padded, group):
        parts = [torch.empty(padded.shape, dtype=padded.dtype) for _ in range(world)]
        dist.all_gather(parts, padded.cpu(), group=group)
        gathered = [g.to(local.device) for g in parts]
    else:
        gathered = [torch.empty_like(padded) for _ in range(world)]
        dist.all_gather(gathered, padded, group=group)
    return torch.cat([gathered[g][..., :bands.size(g), :] for g in range(world)], dim=-2)


def source_band_for_proc_rows(src_ra_shape: Tuple[int, int], src_transform: Affine, ref_transform: Affine,
                              proc_rows: Tuple[int, int]) -> Tuple[int, int]:
    """
    Source rows whose pixel CENTRES fall inside proc-grid rows ``[proc_rows[0], proc_rows[1])`` (north-up grids).  With
    an integer, aligned ratio these are exactly the ``ratio * n`` source rows under the band.
    """
    import math
    sy = ref_transform.e / src_transform.e
    oy = (ref_transform.f - src_transform.f) / src_transform.e
    r0 = max(int(math.ceil(sy * proc_rows[0] + oy - 0.5)), 0)
    r1 = min(int(math.ceil(sy * proc_rows[1] + oy - 0.5)), src_ra_shape[0])
    return r0, max(r1, r0)


def fit_row_window(bands: RowBands, rank: int, halo: int, reach: int = 2) -> Tuple[int, int, int, int]:
    """
    Proc-grid rows of the sharded proc_crs = ref path for ``rank``: ``(lo, hi, plo, phi)``.  ``[lo, hi)`` are the rows the
    rank holds for the fit (its band extended by ``halo`` rows, clipped to the raster); ``[plo, phi)`` are the rows whose
    parameters it needs for the up-sampler (its band plus the ``reach`` rows of tap support on either side, clipped:
    2 for the 4-tap methods, 3 for lanczos).  Every kept row is at least ``halo - reach`` rows away from a cut edge of
    the held window -- the distance over which window sums (and the in-painting search) are affected by the cut --
    unless that edge is the raster's own.
    """
    a, b = bands.band(rank)
    hp = bands.starts[-1]
    lo, hi = max(a - halo, 0), min(b + halo, hp)
    plo, phi = max(a - reach, 0), min(b + reach, hp)
    return lo, hi, plo, phi


# ---------------------------------------------------------------------------------------------------------------------
# whole-block statistics of a sharded block
# ---------------------------------------------------------------------------------------------------------------------
def _all_gather_bytes(local: torch.Tensor, group=None) -> torch.Tensor:
    """ ``[world * n]`` uint8 tensor holding every rank's ``[n]`` uint8 tensor, in rank order. """
    world = dist.get_world_size(group)
    if _host_staged(local, group):
        parts = [torch.empty(local.shape, dtype=local.dtype) for _ in range(world)]
        dist.all_gather(parts, local.cpu(), group=group)
        return torch.cat(parts).to(local.device)
    out = torch.empty(world * local.numel(), dtype=local.dtype, device=local.device)
    if local.is_cuda:
        dist.all_gather_into_tensor(out, local, group=group)
        return out
    try:
        dist.all_gather_into_tensor(out, local, group=group)
    except (RuntimeError, NotImplementedError):          # back ends without the flat variant
        parts = [torch.empty_like(local) for _ in range(world)]
        dist.all_gather(parts, local, group=group)
        out = torch.cat(parts)
    return out


class NativeBlockNorm:
    """ The three accumulate / merge passes of ``hb_block_norm_partial`` / ``hb_block_norm_merge`` on device planes. """
    _sizes: dict = {}

    def __init__(self, src_local: torch.Tensor, src_nodata, ref_local: torch.Tensor, ref_nodata, n_local_max: int,
                 n_total: int, rank: int):
        from homonim_b200 import _native
        from homonim_b200 import kernel_model as km
        self._km, self._lib = km, _native.lib()
        if src_local.dtype != torch.float32 or ref_local.dtype != torch.float32:
            raise ValueError('block statistics are taken on float32 planes')
        if not (src_local.is_contiguous() and ref_local.is_contiguous()):
            raise ValueError('block statistics need contiguous planes (row ranges of a plane are fine)')
        self.src, self.ref = src_local, ref_local
        self.n = int(src_local.numel())
        self.n_local_max, self.n_total, self.rank = int(n_local_max), int(n_total), int(rank)
        self.s_nd, self.r_nd = km._nodata_args(src_nodata), km._nodata_args(ref_nodata)
        key = (self.n_local_max, self.n_total)
        if key not in NativeBlockNorm._sizes:
            NativeBlockNorm._sizes[key] = (int(self._lib.hb_block_norm_shard_workspace_bytes(*key)),
                                           int(self._lib.hb_block_norm_message_bytes(*key)))
        self.ws_bytes, self.msg_bytes = NativeBlockNorm._sizes[key]
        self.work = torch.empty(self.ws_bytes, dtype=torch.uint8, device=src_local.device)
        self.norm = torch.empty(2, dtype=torch.float64, device=src_local.device)

    def partial(self, level: int) -> torch.Tensor:
        km = self._km
        km._call('hb_block_norm_partial', level, self.src.data_ptr() if self.n else None, self.s_nd[0], self.s_nd[1],
                 self.ref.data_ptr() if self.n else None, self.r_nd[0], self.r_nd[1], self.n, self.n_local_max,
                 self.n_total, self.work.data_ptr(), self.ws_bytes, km._stream())
        return self.work[:self.msg_bytes]

    def merge(self, level: int, gathered: torch.Tensor, world: int):
        km = self._km
        km._call('hb_block_norm_merge', level, gathered.data_ptr(), world, self.rank, self.n_local_max, self.n_total,
                 self.work.data_ptr(), self.ws_bytes, self.norm.data_ptr(), km._stream())


def block_norm_sharded(src_local: torch.Tensor, src_nodata, ref_local: torch.Tensor, ref_nodata, group=None,
                       backend=NativeBlockNorm, n_local_max: Optional[int] = None, n_total: Optional[int] = None
                       ) -> torch.Tensor:
    """
    ``KernelModel._fit_block_norm`` (kernel_model.py:216-229) of a block whose rows are spread over the ranks: every rank
    passes ITS rows of the two planes and gets the two float64 statistics of the whole block -- identical on all ranks,
    and (blocks up to 2^28 pixels) identical to the unsharded ``hb_block_norm``, numpy's pairwise float32 ``np.std``
    included.  Three passes, each followed by one all-gather of the pass's message (counts, sums, histograms, the shard's
    first / last valid pixels and its pairwise-leaf sums; ~131 KB + 1/8 byte per pixel) and a merge in rank order.
    ``n_local_max`` / ``n_total``: pixels of the largest shard / of the whole block (callers that partition the raster
    know them; otherwise one small all-reduce finds them).  ``backend`` supplies the two native steps (the CPU tests
    substitute a numpy stand-in to exercise this protocol over gloo).
    """
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    n = int(src_local.numel())
    if n_local_max is None or n_total is None:
        if world > 1:
            counts = torch.tensor([n, n], dtype=torch.int64, device=src_local.device if not _host_staged(src_local, group)
                                  else 'cpu')
            total, largest = counts[:1].clone(), counts[1:].clone()
            dist.all_reduce(total, op=dist.ReduceOp.SUM, group=group)
            dist.all_reduce(largest, op=dist.ReduceOp.MAX, group=group)
            n_total, n_local_max = int(total.item()), int(largest.item())
        else:
            n_total = n_local_max = n
    state = backend(src_local, src_nodata, ref_local, ref_nodata, max(int(n_local_max), 1), max(int(n_total), 1), rank)
    for level in range(3):
        msg = state.partial(level)
        gathered = _all_gather_bytes(msg, group) if world > 1 else msg
        state.merge(level, gathered, world)
    return state.norm


# ---------------------------------------------------------------------------------------------------------------------
# halo rows received in place
# ---------------------------------------------------------------------------------------------------------------------
def alloc_with_halo(bands: RowBands, rank: int, halo: int, width: int, dtype, device) -> Tuple[torch.Tensor, int]:
    """
    An uninitialised ``[rows of bands.with_halo(rank, halo), width]`` plane and the number of halo rows on top: fill
    rows ``[top, top + bands.size(rank))`` with the rank's own rows, then `exchange_halos_inplace` fills the rest.
    """
    a, _ = bands.band(rank)
    lo, hi = bands.with_halo(rank, halo)
    return torch.empty((hi - lo, width), dtype=dtype, device=device), a - lo


def exchange_halos_inplace(ext: torch.Tensor, bands: RowBands, halo: int, group=None) -> None:
    """
    Fill the halo rows of ``ext`` (``[..., rows of bands.with_halo(rank, halo), width]``, own rows already in place) from
    the row-band neighbours, point to point, receiving straight into ``ext``: nothing but the halo rows moves.
    """
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    if world == 1 or halo == 0:
        return
    a, b = bands.band(rank)
    lo, hi = bands.with_halo(rank, halo)
    if ext.shape[-2] != hi - lo:
        raise ValueError(f'`ext` must hold the {hi - lo} rows of the band with its halo, not {ext.shape[-2]}')
    sends, recvs = [], []
    for peer in _halo_peers(bands, rank, halo):
        pa, pb = bands.band(peer)
        plo, phi = bands.with_halo(peer, halo)
        s0, s1 = max(a, plo), min(b, phi)                # rows of mine that the peer needs
        if s1 > s0:
            sends.append((ext[..., s0 - lo:s1 - lo, :], peer))
        r0, r1 = max(pa, lo), min(pb, hi)                # rows of the peer that I need
        if r1 > r0:
            recvs.append((ext[..., r0 - lo:r1 - lo, :], peer))
    _run_p2p(sends, recvs, group)


# ---------------------------------------------------------------------------------------------------------------------
# the two sharded regimes
# ---------------------------------------------------------------------------------------------------------------------
class _RefspaceShard(NamedTuple):
    """ State between the two stages of `fuse_refspace_sharded` (one band of one rank). """
    model: object
    src_t: torch.Tensor
    src_local: RasterArray
    ref_ra: RasterArray
    ref_t: torch.Tensor
    bands: RowBands
    group: object
    src_ds_local: torch.Tensor
    ds_done: object            # CUDA event: the down-sampling has finished (None on the host back end)


def fuse_refspace_sharded_begin(model, src_local: RasterArray, ref_ra: RasterArray, bands: RowBands, group=None
                                ) -> _RefspaceShard:
    """
    First stage of `fuse_refspace_sharded`: the down-sampling of this rank's source rows (the first of the band's two
    streaming kernels; no communication).  Callers with several bands enqueue this stage for ALL bands first and the
    second stages afterwards: the GPU then always has a streaming kernel queued while the host issues the small kernels
    and exchanges of the second stages (with a slab of a few thousand rows per rank those are host-paced, not GPU-paced).
    """
    from homonim_b200 import kernel_model as km
    from homonim_b200.enums import Resampling
    rank = _rank(group)
    a, b = bands.band(rank)
    src_t = km._to_device(src_local.array)
    ref_t = km._as_f32_plane(km._to_device(ref_ra.array), ref_ra.nodata).contiguous()
    local_tf = ref_ra.transform * Affine.translation(0, a)
    # (a footprint statistic is exact here for the reason `average` is: every processing row's footprint lies inside
    # the source rows `source_band_for_proc_rows` gives this rank)
    stat = km._STAT_METHODS.get(Resampling.coerce(model._downsampling))
    if stat is not None:
        src_ds_local = km._resample_stat(src_t, src_local.transform, src_local.nodata, (b - a, ref_ra.width), local_tf,
                                         stat)
    else:
        src_ds_local = km._downsample_average(src_t, src_local.transform, src_local.nodata, (b - a, ref_ra.width),
                                              local_tf)
    ds_done = None
    if src_ds_local.is_cuda:
        ds_done = torch.cuda.Event()
        ds_done.record(km.current_stream())
    return _RefspaceShard(model, src_t, src_local, ref_ra, ref_t, bands, group, src_ds_local, ds_done)


def fuse_refspace_sharded_end(shard: _RefspaceShard, out=None, apply_stream=None) -> Tuple[RasterArray, RasterArray]:
    """
    Second stage of `fuse_refspace_sharded`: block statistics merged over the ranks, halo rows, fit, up-sample + apply.

    The stage may run on a different stream than the first (it waits for the down-sampling's event), and
    ``apply_stream`` (optional) receives the final up-sample + apply kernel.  That lets a caller keep the two STREAMING
    kernels of every band on low-priority streams and this stage's small kernels and exchanges on a high-priority one:
    the block scheduler dispatches pending kernels of equal priority in launch order, so at equal priority a small
    kernel launched behind another band's streaming kernel only runs once that kernel has handed out all its CTAs
    (measured: the stages then simply add up); with priorities it slips in between.
    """
    from homonim_b200 import kernel_model as km
    from homonim_b200.enums import Model
    model, src_t, src_local, ref_ra, ref_t, bands, group, src_ds_local, ds_done = shard
    rank = _rank(group)
    a, b = bands.band(rank)
    nan = float('nan')
    if ds_done is not None:
        cur = km.current_stream()
        cur.wait_event(ds_done)
        src_ds_local.record_stream(cur)
    # whole-block statistics from per-rank accumulators
    norm = None
    if model.model == Model.gain_blk_offset:
        widest = max(bands.size(g) for g in range(len(bands.starts) - 1)) * ref_ra.width
        norm = block_norm_sharded(src_ds_local, nan, ref_t[a:b], ref_ra.nodata, group, n_local_max=widest,
                                  n_total=ref_ra.height * ref_ra.width)
    # halo rows of the down-sampled plane, point to point
    inpaint = model.model == Model.gain_offset and model._r2_inpaint_thresh is not None
    reach = up_reach(model._upsampling)
    halo = halo_rows(model.kernel_shape, proc_crs_ref=True, inpaint=inpaint, reach=reach)
    lo, hi, plo, phi = fit_row_window(bands, rank, halo, reach)
    src_ds, _ = exchange_halos(src_ds_local, bands, halo, group)
    # fit the rows my source rows' spline taps touch, inside the held window
    params = model._fit_planes(src_ds, nan, ref_t[lo:hi], ref_ra.nodata, norm=norm, rows=(plo - lo, phi - plo))
    param_ra = RasterArray(params, ref_ra.crs, ref_ra.transform * Affine.translation(0, plo), nodata=nan)
    # apply to my source rows
    src_ra = RasterArray(src_t, src_local.crs, src_local.transform, nodata=src_local.nodata)
    if apply_stream is not None and params.is_cuda:
        fitted = torch.cuda.Event()
        fitted.record(km.current_stream())
        apply_stream.wait_event(fitted)
        params.record_stream(apply_stream)
        with km.on_stream(apply_stream):
            corr_local = model.apply(src_ra, param_ra, out=out)
    else:
        corr_local = model.apply(src_ra, param_ra, out=out)
    return corr_local, param_ra


def fuse_refspace_sharded(model, src_local: RasterArray, ref_ra: RasterArray, bands: RowBands, group=None, out=None
                          ) -> Tuple[RasterArray, RasterArray]:
    """
    proc_crs = ref fit + apply of ONE band of a raster that is sharded by rows (configuration C5a).

    ``src_local`` holds this rank's source rows (its transform already points at its first row); ``ref_ra`` is the
    whole (replicated: it is 1 / ratio^2 of the source) reference band on the proc grid; ``bands`` partitions the
    proc-grid rows.  Returns ``(corr_local, param_ra)``: the corrected rows of this rank and the parameters of the
    proc-grid rows they depend on (this rank's band plus the 2 rows of tap support on either side, 3 for lanczos;
    ``param_ra.transform`` points at them).  ``out`` (optional): float32 CUDA tensor to receive the corrected rows.

    Per rank: down-sample own rows (`fuse_refspace_sharded_begin`) -> block statistics over own proc rows, merged by
    `block_norm_sharded` (gain-blk-offset) -> halo rows of the down-sampled source from the neighbours -> fit of the rows
    the up-sampler needs -> up-sample + apply on own source rows (`fuse_refspace_sharded_end`).  No rank reads pixels
    outside its band + halo.
    """
    return fuse_refspace_sharded_end(fuse_refspace_sharded_begin(model, src_local, ref_ra, bands, group), out=out)


def fit_same_grid_sharded(model, src_local: torch.Tensor, src_nodata, ref_local: torch.Tensor, ref_nodata,
                          bands: RowBands, group=None) -> torch.Tensor:
    """
    Same-grid fit of a raster sharded by rows: halo exchange of ``kh // 2`` rows of both planes with the row-band
    neighbours (+ 100 with R2 in-painting), whole-block statistics merged over the ranks for gain-blk-offset, fit of the
    rank's own rows inside the extended band.  Returns the ``[2|3, own rows, W]`` parameters.  (Copies the band into the
    extended plane; callers that own their buffers use `alloc_with_halo` + `fit_apply_same_grid_sharded`.)
    """
    from homonim_b200.enums import Model
    halo = halo_rows(model.kernel_shape, proc_crs_ref=False,
                     inpaint=(model.model == Model.gain_offset and model._r2_inpaint_thresh is not None))
    rank = dist.get_rank(group)
    norm = None
    if model.model == Model.gain_blk_offset:
        width = int(src_local.shape[-1])
        norm = block_norm_sharded(src_local.contiguous(), src_nodata, ref_local.contiguous(), ref_nodata, group,
                                  n_local_max=max(bands.size(g) for g in range(len(bands.starts) - 1)) * width,
                                  n_total=bands.starts[-1] * width)
    src_ext, top = exchange_halos(src_local, bands, halo, group)
    ref_ext, _ = exchange_halos(ref_local, bands, halo, group)
    return model._fit_planes(src_ext.contiguous(), src_nodata, ref_ext.contiguous(), ref_nodata, norm=norm,
                             rows=(top, bands.size(rank)))


def fit_apply_same_grid_sharded(model, src_ext: torch.Tensor, src_nodata, ref_ext: torch.Tensor, ref_nodata,
                                bands: RowBands, group=None, out=None) -> torch.Tensor:
    """
    Same-grid fit + apply of ONE band of a raster sharded by rows (configuration C5b: source and reference on one grid).

    ``src_ext`` / ``ref_ext``: float32 planes from `alloc_with_halo` (halo = `halo_rows(kernel_shape, False, False)`) with
    this rank's own rows in place.  The halo rows are received from the neighbours in place, the block statistics of
    gain-blk-offset are merged over the ranks, and one kernel fits the rank's rows and writes the corrected pixels
    (``hb_fit_apply_same_grid_rows``).  Returns the corrected ``[own rows, W]`` plane (``out`` when given).
    """
    from homonim_b200.enums import Model
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    halo = halo_rows(model.kernel_shape, proc_crs_ref=False, inpaint=False)
    a, b = bands.band(rank)
    lo, _ = bands.with_halo(rank, halo)
    top, n_local = a - lo, b - a
    norm = None
    if model.model == Model.gain_blk_offset:
        width = int(src_ext.shape[-1])
        norm = block_norm_sharded(src_ext[top:top + n_local], src_nodata, ref_ext[top:top + n_local], ref_nodata, group,
                                  n_local_max=max(bands.size(g) for g in range(len(bands.starts) - 1)) * width,
                                  n_total=bands.starts[-1] * width)
    if dist.is_initialized():
        exchange_halos_inplace(src_ext, bands, halo, group)
        exchange_halos_inplace(ref_ext, bands, halo, group)
    return model._fit_apply_rows(src_ext, src_nodata, ref_ext, ref_nodata, top, n_local, norm=norm, out=out)
