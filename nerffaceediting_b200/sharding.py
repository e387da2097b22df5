"""Multi-GPU sharding of the render path: one process per GPU, no collective inside the render.

Rays are independent given planes + decoder weights (SURVEY.md §8e); the only cross-ray coupling in the
reference is the depth clamp's min/max over ALL sample depths (ray_marcher.py:49-50,93-94).  So:

  * batch-first: when the batch has at least one item per rank, each rank renders whole items (a plane set
    then lives on exactly one GPU);
  * ray blocks: otherwise every rank renders a contiguous block of the rays of every item, with the plane
    sets replicated (25-50 MB per item);
  * each rank renders with the clamp deferred, the 2-float depth range is all-reduced (MIN / MAX), the clamp
    applied, and ONE all-gather of the packed [rgb | seg | depth | wsum] maps (49 floats per ray) rebuilds
    the full images on every rank.  That all-gather is the only data-path collective.

The reference has no counterpart (its renderer is single-device; training is plain data parallelism,
train.py:32-52), so this module is the north-star's addition, not a port.
"""
import torch
import torch.distributed as dist


def partition(n_batch, n_rays, world, rank):
    """(axis, lo, hi, padded_share): which slice this rank renders.  axis 'batch' splits items, 'rays' splits
    the ray axis.  Shares are ceil-divided, so trailing ranks may get fewer (or zero) units; padded_share is
    the common all-gather size."""
    if world <= 1:
        return "batch", 0, n_batch, n_batch
    if n_batch >= world:
        share = -(-n_batch // world)
        lo = min(rank * share, n_batch)
        return "batch", lo, min(lo + share, n_batch), share
    share = -(-n_rays // world)
    lo = min(rank * share, n_rays)
    return "rays", lo, min(lo + share, n_rays), share


def pack_maps(rgb, seg, depth, wsum):
    """[N,R,32] [N,R,15]|None [N,R,1] [N,R,1] -> [N,R,49|34]."""
    parts = [rgb] + ([seg] if seg is not None else []) + [depth, wsum]
    return torch.cat(parts, dim=-1)


def unpack_maps(packed, has_seg):
    c = packed.shape[-1]
    seg_dim = c - 34 if has_seg else 0
    rgb = packed[..., :32]
    seg = packed[..., 32:32 + seg_dim] if has_seg else None
    return rgb, seg, packed[..., 32 + seg_dim:33 + seg_dim], packed[..., 33 + seg_dim:34 + seg_dim]


def _all_gather(packed_padded, group):
    world = dist.get_world_size(group)
    out = torch.empty((world,) + tuple(packed_padded.shape), dtype=packed_padded.dtype, device=packed_padded.device)
    if dist.get_backend(group) == "nccl":
        dist.all_gather_into_tensor(out.view(-1), packed_padded.reshape(-1), group=group)
    else:
        _gloo_all_gather(out, packed_padded.contiguous(), group)
    return out


def _gloo_all_gather(full, packed, group):
    """gloo (tests, CPU boxes): list-form all_gather; it has no CUDA all_gather, so device tensors go through the host."""
    world = dist.get_world_size(group)
    if packed.is_cuda:
        host = packed.cpu()
        chunks = [torch.empty_like(host) for _ in range(world)]
        dist.all_gather(chunks, host, group=group)
        full.view((world,) + tuple(packed.shape)).copy_(torch.stack(chunks))
    else:
        dist.all_gather(list(full.view((world,) + tuple(packed.shape)).unbind(0)), packed, group=group)


def _all_gather_into(full, packed, group):
    if dist.get_backend(group) == "nccl":
        dist.all_gather_into_tensor(full, packed, group=group)
    else:
        _gloo_all_gather(full, packed, group)


class PendingMaps:
    """Result of a sharded render whose all-gather may still be running on the communication stream.  `wait()` makes the
    current stream wait for it and returns (rgb, seg|None, depth, wsum) — views of ONE gathered buffer that the next-but-one
    call on the same ShardedRenderer will overwrite."""

    def __init__(self, full, has_seg, event):
        self._full, self._has_seg, self._event = full, has_seg, event

    def wait(self):
        if self._event is not None:
            torch.cuda.current_stream().wait_event(self._event)
            self._event = None
        return unpack_maps(self._full, self._has_seg)


class ShardedRenderer:
    """render_sharded with the collective off the critical path: the all-gather of step i runs on a communication stream out
    of a 2-deep ring of packed buffers while the caller already renders step i+1 (bench.py N > 1; DESIGN.md §1e).
    `local_batch=True` is the batch-first weak-scaling form: every rank passes ITS OWN items (a plane set then lives on exactly
    one GPU, SURVEY.md §8e) and the gathered maps cover world x local batch items in rank order."""

    def __init__(self, renderer, group=None, overlap=True):
        self.renderer, self.group, self.overlap = renderer, group, overlap
        self._ring, self._events, self._i, self._stream = {}, {}, 0, None
        self.last_packed = None          # this rank's packed [rgb|seg|depth|wsum] maps of the latest local_batch call

    def __call__(self, norm_planes, planes, decoder, ray_origins, ray_directions, rendering_options, local_batch=False):
        _no_geometry_only(rendering_options)
        world = dist.get_world_size(self.group) if (dist.is_available() and dist.is_initialized()) else 1
        if not local_batch or world == 1:
            out = render_sharded(self.renderer, norm_planes, planes, decoder, ray_origins, ray_directions, rendering_options, group=self.group)
            return PendingMaps(pack_maps(*out), out[1] is not None, None)
        from . import ops
        dev = ray_origins.device
        n, r = ray_origins.shape[0], ray_origins.shape[1]
        rgb, seg, depth, wsum, minmax = self.renderer._render(norm_planes, planes, decoder, ray_origins, ray_directions, rendering_options,
                                                              defer_clamp=True)
        if rendering_options.get('nfe_deterministic', False):
            # parity mode: every rank's sample depths span the same table, the local range IS the global one
            depth = ops.finish_depth(depth, minmax)
        else:
            lo_hi = torch.stack([minmax[0], -minmax[1]])
            dist.all_reduce(lo_hi, op=dist.ReduceOp.MIN, group=self.group)
            depth = ops.finish_depth(depth, torch.stack([lo_hi[0], -lo_hi[1]]))
        has_seg = seg is not None
        c = 34 + (seg.shape[-1] if has_seg else 0)
        slot = self._i & 1
        self._i += 1
        key = (slot, n, r, c, dev)
        if key not in self._ring:
            self._ring[key] = (torch.empty((n, r, c), device=dev), torch.empty((world * n, r, c), device=dev))
            self._events[key] = torch.cuda.Event()
            self._events[key].record(torch.cuda.current_stream())
        packed, full = self._ring[key]
        main = torch.cuda.current_stream()
        main.wait_event(self._events[key])                       # the all-gather that last read this slot (two calls ago) is done
        torch.cat([rgb] + ([seg] if has_seg else []) + [depth, wsum], dim=-1, out=packed)
        self.last_packed = packed
        if not self.overlap:
            _all_gather_into(full, packed, self.group)
            return PendingMaps(full, has_seg, None)
        if self._stream is None:
            self._stream = torch.cuda.Stream(device=dev)
        ready = torch.cuda.Event()
        ready.record(main)
        with torch.cuda.stream(self._stream):
            self._stream.wait_event(ready)
            _all_gather_into(full, packed, self.group)
            self._events[key].record(self._stream)
        return PendingMaps(full, has_seg, self._events[key])

    def drain(self):
        """Make the current stream wait for every all-gather issued so far (end of a timed region)."""
        if self._stream is not None:
            torch.cuda.current_stream().wait_stream(self._stream)


def _no_geometry_only(rendering_options):
    if rendering_options.get('nfe_geometry_only', False):
        raise NotImplementedError("rendering_options['nfe_geometry_only'] is not built for the sharded renderer")


def render_sharded(renderer, norm_planes, planes, decoder, ray_origins, ray_directions, rendering_options, group=None,
                   render_local=None, finish=None, force_sharded_path=False):
    """Sharded forward of ImportanceRenderer (norm_planes=None) / DisentangledImportanceRenderer.
    Every rank passes the full inputs and receives the full outputs (rgb, seg|None, depth, wsum).
    `render_local` / `finish` are injection points for tests; by default they call the renderer's deferred-clamp
    entry and nfe_finish_depth.  force_sharded_path=True takes the sharded code path (deferred clamp, range reduction,
    pack / pad / all-gather / unpack) even in a world of one — what a single-GPU box can test of it."""
    _no_geometry_only(rendering_options)
    initialized = dist.is_available() and dist.is_initialized()
    if (not initialized or dist.get_world_size(group) == 1) and not (force_sharded_path and initialized):
        return renderer._render(norm_planes, planes, decoder, ray_origins, ray_directions, rendering_options)
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    n, r = ray_origins.shape[0], ray_origins.shape[1]
    axis, lo, hi, share = partition(n, r, world, rank)
    if render_local is None:
        def render_local(np_, p_, o_, d_):
            return renderer._render(np_, p_, decoder, o_, d_, rendering_options, defer_clamp=True)
    if finish is None:
        from . import ops
        finish = ops.finish_depth

    if axis == "batch":
        sl = slice(lo, hi)
        plane_sl = sl if planes.shape[0] == n else slice(None)        # a shared (batch-1) plane set is replicated
        args = (norm_planes[plane_sl] if norm_planes is not None else None, planes[plane_sl], ray_origins[sl], ray_directions[sl])
    else:
        args = (norm_planes, planes, ray_origins[:, lo:hi].contiguous(), ray_directions[:, lo:hi].contiguous())
    rgb, seg, depth, wsum, minmax = render_local(*args)

    # depth clamp over the samples of ALL ranks
    lo_hi = torch.stack([minmax[0], -minmax[1]])
    if hi <= lo:                                                        # an idle rank must not pollute the range
        lo_hi = torch.full_like(lo_hi, float("inf"))
    dist.all_reduce(lo_hi, op=dist.ReduceOp.MIN, group=group)
    if hi > lo:
        depth = finish(depth, torch.stack([lo_hi[0], -lo_hi[1]]))

    has_seg = seg is not None
    packed = pack_maps(rgb, seg, depth, wsum)
    c = packed.shape[-1]
    if axis == "batch":
        padded = packed.new_zeros((share, r, c))
        padded[:hi - lo] = packed
        full = _all_gather(padded, group).reshape(world * share, r, c)[:n]
    else:
        padded = packed.new_zeros((n, share, c))
        padded[:, :hi - lo] = packed
        full = _all_gather(padded, group).permute(1, 0, 2, 3).reshape(n, world * share, c)[:, :r]
    return unpack_maps(full.contiguous(), has_seg)
