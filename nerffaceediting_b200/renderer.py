"""Drop-in ImportanceRenderer / DisentangledImportanceRenderer
(reference: training/volumetric_rendering/renderer.py).

Call signatures, return shapes, attributes (`ray_marcher`, `plane_axes`) and helper methods are the
reference's; the work runs in libnfe_b200.so.  When the decoder is one of the reference's three
(recognised by structure, see ops.describe_decoder) the whole forward is the fused CUDA path and no
per-sample tensor is materialised; any other decoder callable still works through the stage kernels
(gather -> decoder(...) -> composite / resample / merge).

Extra keys read from `rendering_options` (all optional; defaults reproduce the reference):
  nfe_deterministic  False  no stratified jitter and u = linspace(0,1,S_f): the parity mode.  The
                            reference has no such switch (renderer.py:180-190,210-211); its always-on
                            jitter is drawn here from an in-kernel Philox stream seeded from torch's
                            CUDA generator (statistically, not bitwise, equal to torch.rand).
  nfe_precision    'bf16x3' arithmetic of the decoder MLPs: 'bf16x3' (tcgen05 tensor cores, three bf16 MMAs per product with
                            fp32 accumulation, fp32-grade: meets the path's 1e-4 tolerance; the default, overridable with
                            $NFE_DEFAULT_PRECISION), 'fp32' (FFMA on the CUDA cores) or 'bf16' (tensor cores, 1e-2).
  nfe_single_gather  True   disentangled renderer, tensor-core modes: when the de-normalised planes are known to be
                            norm*scale+shift per channel (they came from normalize_plane / denormalize_plane of this
                            package), gather only the normalised planes and rebuild the other features from the statistics.
  nfe_sigma_only     False  run_model only: return {'sigma'} alone (shape extraction gen_samples.py:184-222, density regulariser
                            loss.py:310-331); with the disentangled decoder the appearance net and its gather are skipped.
  nfe_image_layout   False  return (feature_image [N,32,H,W], seg_image [N,15,H,W], depth_image [N,1,H,W], weights [N,R,1]) —
                            what triplane.py:122-125 builds with three permute+reshape+contiguous passes — written in that
                            layout by the compositing kernel itself.
  nfe_cache_planes   False  keep the channel-last staging of the planes between calls (video sweeps).
  nfe_geometry_only  False  render geometry alone: forward returns (None, seg, depth, wsum) (disentangled) or (None, depth, wsum),
                            bit-identical to the full render's maps, without the appearance branch: no colours are decoded or
                            composited, the per-sample records shrink to a third, and the disentangled decoder reads only the
                            normalised planes (the raw ones are neither staged nor gathered); a render with draws is split into
                            workspace chunks where the full render would be, so it draws the same samples.  Inference only; the staged path
                            (other decoders) honours the same outputs but saves nothing.

Instances hold no state of their own beyond the reference's attributes, so objects unpickled from
reference checkpoints (which skip __init__, SURVEY.md §7.9) work.
"""
import os
from typing import NamedTuple

import torch
import torch.nn as nn

from . import math_utils, ops
from .ray_marcher import MipRayMarcher2, SegMipRayMarcher2


class FieldPlan(NamedTuple):
    """How the fused forward of one render or run_model call reads the tri-planes (made by field_plan)."""
    kind: int
    seq_a: object
    seq_b: object           # None for the OSG decoder
    precision: int
    geo_only: bool          # density-only query, disentangled decoder on the tensor cores: the appearance net and its planes are skipped
    geometry: bool          # geometry-only render (rendering_options['nfe_geometry_only']): no colours; disentangled: geo_net on the normalised planes
    affine: object          # (scale [K,96], shift [K,96]) under the single-gather identity, else None
    sources: object         # training under the identity: (scale_src, shift_src), the autograd inputs of the affine pair, else None
    stage_norm: bool        # which plane sets are staged channel-last
    stage_denorm: bool
    library_gemm: bool      # NFE_BWD_LIBRARY_GEMM=1: the backward runs the decoder MLPs on library GEMMs (autograd._FieldBackward)
    path: object            # (what, path) for ops.note_path, or None


def field_plan(what, desc, norm_planes, planes, opts, batch, per_item, grad, sigma_only=False, geometry=False):
    """Decide the fused forward of one call: what = 'render' (per_item rays per batch item) or 'run_model' (per_item points),
    desc = ops.describe_decoder(decoder), grad = whether the call is differentiable, geometry = a geometry-only render
    (inference only).  It reads the options, the environment and the plane registries and calls no kernel, so it runs on CPU
    tensors as well."""
    kind, seq_a, seq_b = desc
    precision = ops.precision_of(opts)
    disentangled_tc = kind == ops.DEC_DISENTANGLED and precision != ops.PRECISIONS['fp32']
    geo_only = sigma_only and disentangled_tc
    # geometry-only render, disentangled decoder: geo_net reads the normalised planes alone (every precision), so the raw
    # planes are neither staged nor gathered and their provenance is not needed
    norm_only = geometry and kind == ops.DEC_DISENTANGLED
    library_gemm = os.environ.get("NFE_BWD_LIBRARY_GEMM", "0") == "1"
    if what == "render":
        s_c, s_f = opts['depth_resolution'], opts['depth_resolution_importance']
        per_item *= min(s_c, s_f if s_f > 0 else s_c)
    # The field kernel keeps the statistics of at most two batch items per 128-sample tile, so the single-gather identity needs
    # every item to hold at least one tile's worth of samples in each pass (always true for renders; tiny point queries simply
    # read both plane sets).
    single = disentangled_tc and opts.get('nfe_single_gather', True) and per_item >= 128
    affine = sources = None
    if not grad:
        # planes known to be norm*scale + shift per channel (normalize_plane / denormalize_plane made them): gather the
        # normalised planes only and rebuild the de-normalised features from the statistics
        if single and not geo_only and not norm_only:
            affine = ops.provenance(norm_planes, planes)
        path = (what, "single-gather" if (affine is not None or geo_only) else ("two-gather" if kind == ops.DEC_DISENTANGLED else "one-set"))
        if geometry:
            path = (what, "geometry-only")
    else:
        # In training the identity replaces the gradient into `planes` by gradients into the normalised planes and the
        # statistics `planes` is tied to (normalize_plane: planes is their root; denormalize_plane: planes is their product),
        # which is only the same thing while the autograd graph still has the shape it had when the pair was made: `planes`
        # must carry grad and `norm_planes` must be in the state it was registered in.  A pair with one branch detached
        # afterwards (renderer(norm.detach(), planes), renderer(norm, planes.detach())) takes the two-gather backward, which
        # honours the detach like the reference does.  The library-GEMM cross-check of the backward reads both plane sets.
        src = ops.provenance_sources(norm_planes, planes) if (single and not library_gemm) else None
        if (src is not None and src[0].numel() == src[2].numel() and src[0].numel() in (96, 96 * batch)
                and planes.requires_grad and bool(norm_planes.requires_grad) == src[3]):
            scale_src, eps, shift_src, _ = src
            k = scale_src.numel() // 96
            affine = ((scale_src.detach().reshape(k, 96).float() + eps).contiguous(), shift_src.detach().reshape(k, 96).float().contiguous())
            sources = (scale_src, shift_src)
        path = (what, "training-single-gather" if sources else "training") if what == "render" else None
    # a differentiable run_model stages the raw planes even when geometry-only: its backward returns their gradient in that shape
    return FieldPlan(kind, seq_a, seq_b, precision, geo_only, geometry, affine, sources, kind == ops.DEC_DISENTANGLED,
                     affine is None and not (geo_only and not grad) and not norm_only, library_gemm, path)


def _stage(plan, norm_planes, planes, cache):
    """Channel-last staging of the plane sets `plan` reads: (norm_cl, denorm_cl), None for a set that is not read."""
    norm_cl = ops.planes_channel_last(norm_planes, cache) if plan.stage_norm else None
    denorm_cl = ops.planes_channel_last(planes, cache) if plan.stage_denorm else None
    return norm_cl, denorm_cl


def render_planes(plan, norm_planes, planes, origins, dirs, depths_coarse, u_fine, opts, stochastic, seed, offset, cache=False,
                  image_layout=False, **taps):
    """Fused render forward of inference and of autograd.RenderFunction: stage, build the cfg, ops.render_fwd (taps are its
    finish_depth / return_stages / keep_workspace).  Returns (cfg, norm_cl, denorm_cl, render_fwd's outputs)."""
    norm_cl, denorm_cl = _stage(plan, norm_planes, planes, cache)
    planes_cl = norm_cl if denorm_cl is None else denorm_cl
    if planes_cl.shape[0] not in (1, origins.shape[0]):
        raise RuntimeError(f"planes batch {planes_cl.shape[0]} does not match ray batch {origins.shape[0]}")
    cfg = ops.make_cfg(plan.kind, planes_cl, opts['depth_resolution'], opts['depth_resolution_importance'], opts['box_warp'],
                       opts.get('white_back', False), opts.get('density_noise', 0) or 0.0, stochastic=stochastic, seed=seed, offset=offset,
                       precision=plan.precision, affine=plan.affine)
    cfg.image_layout = int(image_layout)
    cfg.geometry_only = int(plan.geometry)
    return cfg, norm_cl, denorm_cl, ops.render_fwd(cfg, plan.seq_a, plan.seq_b, norm_cl, denorm_cl, origins, dirs, depths_coarse, u_fine, **taps)


def run_model_planes(plan, norm_planes, planes, coords, opts, seed, offset, sigma_only, cache=False):
    """Fused run_model forward of inference and of autograd.RunModelFunction: stage, build the cfg, ops.run_model_fwd.
    Returns (cfg, norm_cl, denorm_cl, run_model_fwd's outputs)."""
    norm_cl, denorm_cl = _stage(plan, norm_planes, planes, cache)
    cfg = ops.make_cfg(plan.kind, norm_cl if denorm_cl is None else denorm_cl, 2, 0, opts['box_warp'], density_noise=opts.get('density_noise', 0) or 0.0,
                       seed=seed, offset=offset, precision=plan.precision, affine=plan.affine)
    return cfg, norm_cl, denorm_cl, ops.run_model_fwd(cfg, plan.seq_a, plan.seq_b, norm_cl, denorm_cl, coords, sigma_only=sigma_only)


def generate_planes():
    """The three plane bases of EG3D (renderer.py:23-37).  With `project_onto_planes` they select
    (x,y), (x,z), (z,x) — the kernels hard-code exactly this projection."""
    return torch.tensor([[[1, 0, 0], [0, 1, 0], [0, 0, 1]],
                         [[1, 0, 0], [0, 0, 1], [0, 1, 0]],
                         [[0, 0, 1], [1, 0, 0], [0, 1, 0]]], dtype=torch.float32)


_CANONICAL_AXES = generate_planes()


def project_onto_planes(planes, coordinates):
    """coordinates [N,M,3] -> [N*n_planes,M,2] plane coordinates (renderer.py:39-53).  Not on the hot path
    (the kernels project in registers); kept for API parity."""
    n, m, _ = coordinates.shape
    n_planes = planes.shape[0]
    coordinates = coordinates.unsqueeze(1).expand(-1, n_planes, -1, -1).reshape(n * n_planes, m, 3)
    inv_planes = torch.linalg.inv(planes).unsqueeze(0).expand(n, -1, -1, -1).reshape(n * n_planes, 3, 3)
    return torch.bmm(coordinates, inv_planes)[..., :2]


def _check_axes(plane_axes):
    if plane_axes is not None and not torch.equal(plane_axes.detach().cpu().float(), _CANONICAL_AXES):
        raise NotImplementedError("sample_from_planes: only the EG3D plane axes of generate_planes() are built into the kernels")


def sample_from_planes(plane_axes, plane_features, coordinates, mode='bilinear', padding_mode='zeros', box_warp=None):
    """plane_features [N,3,C,H,W], coordinates [N,M,3] -> [N,3,M,C]: bilinear, zero padding,
    align_corners=False (renderer.py:55-65)."""
    assert padding_mode == 'zeros'
    if mode != 'bilinear':
        raise NotImplementedError("sample_from_planes: only mode='bilinear' is built")
    _check_axes(plane_axes)
    ops._no_grad_needed(plane_features, coordinates)
    return ops.sample_planes(ops.planes_channel_last(plane_features), coordinates, box_warp)


def sample_from_3dgrid(grid, coordinates):
    """Trilinear 5-D lookup (renderer.py:67-80).  Unused by every caller in the reference; plain ATen."""
    batch_size, n_coords, n_dims = coordinates.shape
    sampled = torch.nn.functional.grid_sample(grid.expand(batch_size, -1, -1, -1, -1),
                                              coordinates.reshape(batch_size, 1, 1, -1, n_dims),
                                              mode='bilinear', padding_mode='zeros', align_corners=False)
    n, c, h, w, d = sampled.shape
    return sampled.permute(0, 4, 3, 2, 1).reshape(n, h * w * d, c)


def _auto_limits(ray_origins, ray_directions, box_warp):
    """'auto' near/far (renderer.py:91-97): box intersection, rays that miss patched with the extrema of
    the valid starts.  The reference syncs on `.item()`; this stays on the device."""
    ray_start, ray_end = math_utils.get_ray_limits_box(ray_origins, ray_directions, box_side_length=box_warp)
    valid = ray_end > ray_start
    inf = torch.full_like(ray_start, float('inf'))
    lo = torch.where(valid, ray_start, inf).min()
    hi = torch.where(valid, ray_start, -inf).max()
    keep = valid | ~valid.any()
    return torch.where(keep, ray_start, lo), torch.where(keep, ray_end, hi)


class ImportanceRenderer(torch.nn.Module):
    _disentangled = False

    def __init__(self):
        super().__init__()
        self.ray_marcher = MipRayMarcher2()
        self.plane_axes = generate_planes()

    # ------------------------------------------------------------------ forward (renderer.py:88-140)
    def forward(self, planes, decoder, ray_origins, ray_directions, rendering_options):
        """planes [N,3,32,H,W] -> (rgb [N,R,32], depth [N,R,1], weights.sum(2) [N,R,1])."""
        rgb, _, depth, wsum = self._render(None, planes, decoder, ray_origins, ray_directions, rendering_options)
        return rgb, depth, wsum

    def _fused_decoder(self, decoder, norm_planes):
        """(kind, net_a, net_b) if `decoder` is one of the reference's three AND matches this renderer's
        calling convention (2-argument OSG for ImportanceRenderer, 3-argument decoders for the
        disentangled renderer); None sends the call down the staged path."""
        desc = ops.describe_decoder(decoder)
        if desc is None or (desc[0] == ops.DEC_OSG) == self._disentangled:
            return None
        if desc[0] == ops.DEC_DISENTANGLED and norm_planes is None:
            return None
        return desc

    def _coarse_depths(self, ray_origins, ray_directions, opts, deterministic):
        n, r, _ = ray_origins.shape
        s_c = opts['depth_resolution']
        seed, offset = (0, 0) if deterministic else ops.philox_state(ray_origins.device)
        # the string test first: comparing a float with 'auto' is fine, a tensor is not
        if isinstance(opts['ray_start'], str) and opts['ray_start'] == opts['ray_end'] == 'auto':
            ray_start, ray_end = _auto_limits(ray_origins, ray_directions, opts['box_warp'])
        else:
            ray_start, ray_end = opts['ray_start'], opts['ray_end']
        depths = ops.sample_stratified(n, r, s_c, ray_origins.device, ray_start, ray_end,
                                       disparity=opts.get('disparity_space_sampling', False),
                                       stochastic=not deterministic, seed=seed, offset=offset)
        return depths, seed, offset

    def _render(self, norm_planes, planes, decoder, ray_origins, ray_directions, opts, defer_clamp=False):
        """Shared forward.  defer_clamp=True (used by sharding.render_sharded) leaves the depth unclamped and also
        returns the device {min,max} of this call's sample depths, to be all-reduced before nfe_finish_depth."""
        if isinstance(self.plane_axes, torch.Tensor):
            self.plane_axes = self.plane_axes.to(ray_origins.device)       # as renderer.py:89
        if not ray_origins.is_cuda:
            raise RuntimeError("ImportanceRenderer: expected CUDA tensors (this path has no CPU fallback)")
        assert opts['clamp_mode'] == 'softplus', "MipRayMarcher only supports `clamp_mode`=`softplus`!"
        if torch.is_grad_enabled() and (ray_origins.requires_grad or ray_directions.requires_grad):
            # the reference would back-propagate into the cameras (pose optimisation); no caller in the reference does, and
            # silently detaching would be wrong
            raise RuntimeError("ImportanceRenderer: gradients w.r.t. ray_origins / ray_directions are not built; detach the rays")
        deterministic = bool(opts.get('nfe_deterministic', False))
        geometry = bool(opts.get('nfe_geometry_only', False))
        if geometry:
            if defer_clamp:
                raise NotImplementedError("rendering_options['nfe_geometry_only'] is not built for the ray-sharded render")
            params = tuple(decoder.parameters()) if isinstance(decoder, nn.Module) else ()
            if torch.is_grad_enabled() and any(isinstance(t, torch.Tensor) and t.requires_grad for t in (norm_planes, planes, *params)):
                raise RuntimeError("rendering_options['nfe_geometry_only'] is inference-only (it has no backward): "
                                   "call under torch.no_grad() or detach the inputs")
        desc = self._fused_decoder(decoder, norm_planes)
        if desc is None:
            ops.note_path("render", "staged")
            if defer_clamp:
                raise NotImplementedError("a ray-sharded render needs one of the reference's decoders (fused path)")
            rgb, seg, depth, wsum = self._render_staged(norm_planes, planes, decoder, ray_origins, ray_directions, opts, deterministic)
            return (None if geometry else rgb), seg, depth, wsum      # geometry-only: the caller's decoder ran in full, rgb is dropped
        grad = torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in (norm_planes, planes, *decoder.parameters()))
        if grad and defer_clamp:
            raise NotImplementedError("the ray-sharded render is inference-only")
        n, r, _ = ray_origins.shape
        plan = field_plan("render", desc, norm_planes, planes, opts, n, r, grad, geometry=geometry)
        ops.note_path(*plan.path)
        image = bool(opts.get('nfe_image_layout', False)) and not defer_clamp and not grad
        side = int(round(r ** 0.5))
        if image and side * side != r:
            raise RuntimeError("nfe_image_layout needs a square ray grid (RaySampler's res*res rays)")
        depths_coarse, seed, offset = self._coarse_depths(ray_origins, ray_directions, opts, deterministic)
        s_f = opts['depth_resolution_importance']
        u_fine = ops.linspace_table(0, 1, s_f, ray_origins.device) if (s_f > 0 and deterministic) else None
        if grad:
            # differentiable forward (BASELINE config 4): the same fused kernels, workspace kept for autograd.RenderFunction's
            # backward; gradients flow to the plane tensors (or the statistics, under the single-gather identity) and the decoder
            from .autograd import RenderFunction, _decoder_params
            args = (ray_origins.detach().float().contiguous(), ray_directions.detach().float().contiguous(), depths_coarse, u_fine, opts,
                    not deterministic, seed, offset)
            out = RenderFunction.apply(plan, args, norm_planes if plan.stage_norm else None, planes, *(plan.sources or (None, None)),
                                       *_decoder_params(plan.seq_a, plan.seq_b))
            return (out[0], None, out[1], out[2]) if plan.kind == ops.DEC_OSG else out[:4]
        _, _, _, (rgb, seg, depth, wsum, minmax) = render_planes(
            plan, norm_planes, planes, ray_origins, ray_directions, depths_coarse, u_fine, opts, not deterministic, seed, offset,
            cache=bool(opts.get('nfe_cache_planes', False)), image_layout=image, finish_depth=not defer_clamp)
        if defer_clamp:
            return rgb, seg, depth, wsum, minmax
        if image:
            return (None if rgb is None else rgb.view(n, 32, side, side), None if seg is None else seg.view(n, seg.shape[1], side, side),
                    depth.view(n, 1, side, side), wsum)
        return rgb, seg, depth, wsum

    def _render_staged(self, norm_planes, planes, decoder, ray_origins, ray_directions, opts, deterministic):
        """Any decoder callable: the reference's orchestration (renderer.py:99-140,320-363) over the stage
        kernels.  Per-sample tensors are materialised, as in the reference."""
        depths_coarse, _, _ = self._coarse_depths(ray_origins, ray_directions, opts, deterministic)
        n, r, s_c, _ = depths_coarse.shape
        planes_args = (norm_planes, planes) if self._disentangled else (planes,)

        def evaluate(depths, s):
            coords = (ray_origins.unsqueeze(-2) + depths * ray_directions.unsqueeze(-2)).reshape(n, -1, 3)
            dirs = ray_directions.unsqueeze(-2).expand(-1, -1, s, -1).reshape(n, -1, 3)
            out = self.run_model(*planes_args, decoder, coords, dirs, opts)
            col = out['rgb'].reshape(n, r, s, out['rgb'].shape[-1])
            sig = out['sigma'].reshape(n, r, s, 1)
            seg = out['seg'].reshape(n, r, s, out['seg'].shape[-1]) if 'seg' in out else None
            return col, sig, seg

        col_c, sig_c, seg_c = evaluate(depths_coarse, s_c)
        # the stage kernels below have no backward: a decoder whose outputs carry grad must not be silently detached
        ops._no_grad_needed(col_c, sig_c, seg_c)
        s_f = opts['depth_resolution_importance']
        white = opts.get('white_back', False)
        if s_f > 0:
            _, _, _, weights = ops.composite(col_c, sig_c, depths_coarse, seg_c, white)
            depths_fine = self.sample_importance(depths_coarse, weights, s_f, deterministic=deterministic)
            col_f, sig_f, seg_f = evaluate(depths_fine, s_f)
            all_d, all_c, all_g, all_s = ops.unify_samples(depths_coarse, col_c, sig_c, depths_fine, col_f, sig_f, seg_c, seg_f)
            rgb, seg, depth, weights = ops.composite(all_c, all_s, all_d, all_g, white)
        else:
            rgb, seg, depth, weights = ops.composite(col_c, sig_c, depths_coarse, seg_c, white)
        return rgb, seg, depth, weights.sum(2)

    # ------------------------------------------------------------------ run_model (renderer.py:142-148)
    def run_model(self, planes, decoder, sample_coordinates, sample_directions, options):
        """Gather + decode at explicit points -> {'rgb' [N,M,32], 'sigma' [N,M,1]}."""
        return self._run_model(None, planes, decoder, sample_coordinates, sample_directions, options)

    def _run_model(self, norm_planes, planes, decoder, sample_coordinates, sample_directions, options):
        desc = self._fused_decoder(decoder, norm_planes)
        if desc is not None:
            sigma_only = bool(options.get('nfe_sigma_only', False))
            noise = options.get('density_noise', 0) or 0.0
            seed, offset = ops.philox_state(sample_coordinates.device) if noise > 0 else (0, 0)
            grad = torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in (norm_planes, planes, *decoder.parameters()))
            plan = field_plan("run_model", desc, norm_planes, planes, options, *sample_coordinates.shape[:2], grad, sigma_only)
            if grad:
                # differentiable point queries (the density regulariser, loss.py:310-331): autograd.RunModelFunction
                if sample_coordinates.requires_grad:
                    raise RuntimeError("run_model: gradients w.r.t. sample_coordinates are not built (the reference's callers never ask for them)")
                from .autograd import RunModelFunction, _decoder_params
                args = (sample_coordinates.detach().float().contiguous(), options, seed, offset, sigma_only)
                outs = RunModelFunction.apply(plan, args, norm_planes if plan.stage_norm else None, planes, *(plan.sources or (None, None)),
                                              *_decoder_params(plan.seq_a, plan.seq_b))
                keys = ("sigma",) if sigma_only else (("rgb", "sigma") if plan.kind == ops.DEC_OSG else ("rgb", "sigma", "seg"))
                return dict(zip(keys, outs))
            ops._no_grad_needed(sample_coordinates)
            ops.note_path(*plan.path)
            return run_model_planes(plan, norm_planes, planes, sample_coordinates, options, seed, offset, sigma_only,
                                    cache=bool(options.get('nfe_cache_planes', False)))[3]
        axes = self.plane_axes
        feats = sample_from_planes(axes, planes, sample_coordinates, padding_mode='zeros', box_warp=options['box_warp'])
        if self._disentangled:
            norm_feats = sample_from_planes(axes, norm_planes, sample_coordinates, padding_mode='zeros', box_warp=options['box_warp'])
            out = decoder(norm_feats, feats, sample_directions)
        else:
            out = decoder(feats, sample_directions)
        if options.get('density_noise', 0) > 0:
            out['sigma'] += torch.randn_like(out['sigma']) * options['density_noise']
        return out

    # ------------------------------------------------------------------ helpers kept callable
    def sort_samples(self, all_depths, all_colors, all_densities):
        """Sort one sample set by depth (renderer.py:150-155)."""
        d, c, _, s = ops.unify_samples(all_depths, all_colors, all_densities, None, None, None)
        return d, c, s

    def unify_samples(self, depths1, colors1, densities1, depths2, colors2, densities2):
        """cat + sort + gather (renderer.py:157-167)."""
        d, c, _, s = ops.unify_samples(depths1, colors1, densities1, depths2, colors2, densities2)
        return d, c, s

    def sample_stratified(self, ray_origins, ray_start, ray_end, depth_resolution, disparity_space_sampling=False, deterministic=False):
        """depths_coarse [N,M,S,1] (renderer.py:169-192); jitter from Philox unless deterministic."""
        n, m, _ = ray_origins.shape
        seed, offset = (0, 0) if deterministic else ops.philox_state(ray_origins.device)
        return ops.sample_stratified(n, m, depth_resolution, ray_origins.device, ray_start, ray_end, disparity=disparity_space_sampling,
                                     stochastic=not deterministic, seed=seed, offset=offset)

    def sample_importance(self, z_vals, weights, N_importance, deterministic=False):
        """z_vals [N,R,S,1], weights [N,R,S-1,1] -> depths_fine [N,R,N_importance,1], detached
        (renderer.py:194-212)."""
        with torch.no_grad():
            n, r, s, _ = z_vals.shape
            z = z_vals.reshape(n * r, s)
            w = weights.reshape(n * r, -1)
            if deterministic:
                out = ops.importance_resample(z, w, N_importance, u=ops.linspace_table(0, 1, N_importance, z.device))
            else:
                seed, offset = ops.philox_state(z.device)
                out = ops.importance_resample(z, w, N_importance, seed=seed, offset=offset)
        return out.reshape(n, r, N_importance, 1)

    def sample_pdf(self, bins, weights, N_importance, det=False, eps=1e-5):
        """Inverse-CDF sampling of `bins` under `weights` (renderer.py:214-253)."""
        if det:
            u, seed, offset = ops.linspace_table(0, 1, N_importance, bins.device), 0, 0
        else:
            u, (seed, offset) = None, ops.philox_state(bins.device)
        return ops.sample_pdf(bins, weights, N_importance, u=u, seed=seed, offset=offset, eps=eps)


class DisentangledImportanceRenderer(ImportanceRenderer):
    _disentangled = True

    def __init__(self):
        super().__init__()
        self.ray_marcher = SegMipRayMarcher2()

    def forward(self, norm_planes, denorm_planes, decoder, ray_origins, ray_directions, rendering_options):
        """(rgb [N,R,32], seg [N,R,15], depth [N,R,1], weights.sum(2) [N,R,1])  (renderer.py:301-363)."""
        return self._render(norm_planes, denorm_planes, decoder, ray_origins, ray_directions, rendering_options)

    def run_model(self, norm_planes, denorm_planes, decoder, sample_coordinates, sample_directions, options):
        """{'rgb','sigma','seg'} at explicit points (renderer.py:259-287)."""
        return self._run_model(norm_planes, denorm_planes, decoder, sample_coordinates, sample_directions, options)

    def unify_samples(self, depths1, colors1, segs1, densities1, depths2, colors2, segs2, densities2):
        """(renderer.py:288-300); note the (depths, colors, segs, densities) return order."""
        d, c, g, s = ops.unify_samples(depths1, colors1, densities1, depths2, colors2, densities2, segs1, segs2)
        return d, c, g, s
