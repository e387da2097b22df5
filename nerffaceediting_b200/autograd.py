"""Autograd for the render path (BASELINE config 4: training-step forward + backward).

Forward is the same fused CUDA path as inference; its workspace (per-sample densities and {sigma, seg, rgb}
records of both passes) is kept for the backward.  Backward, per SURVEY.md §3.3 / §7.10:

  1. nfe_composite_bwd          ray gradients -> per-sample gradients (warp per ray, CUDA)
  2. nfe_field_bwd / nfe_run_model_bwd   ONE tcgen05 kernel per pass for all three decoders: decoder inputs recomputed from
                                the planes (no [N,3,M,32] tensors were saved), both MLPs back-propagated, parameter gradients
                                accumulated in tensor memory, feature gradients scatter-added into channel-last plane gradients
                                (red.global.add.v4.f32 — atomic, hence ulp-level run-to-run noise like the reference's
                                grid_sampler_2d_backward)
  3. nfe_planes_from_channel_last   back to the reference's [N,3,32,H,W]

NFE_BWD_LIBRARY_GEMM=1 keeps the round-1 cross-check path (nfe_feature_mean_fwd -> decoder MLP backward on torch.addmm ->
nfe_feature_mean_bwd) that the fused kernel is tested against; no product path uses it.

Gradients reach the two plane tensors and the decoder parameters; sample positions carry none (camera labels
are data and depths_fine is detached in the reference, renderer.py:198,211).
"""
import ctypes

import torch
import torch.nn.functional as F

from . import _lib, ops
from .renderer import render_planes, run_model_planes

MAX_ROWS = 1 << 22     # decoder-backward chunk (rows of [M,32] features) to bound the GEMM intermediates


def _mlp(x, seq):
    """FC . Softplus . FC with the FullyConnectedLayer gains (networks_stylegan2.py:114-123)."""
    a, b = seq[0], seq[2]
    h = F.softplus(torch.addmm((a.bias * a.bias_gain).unsqueeze(0), x, (a.weight * a.weight_gain).t()))
    return torch.addmm((b.bias * b.bias_gain).unsqueeze(0), h, (b.weight * b.weight_gain).t())


def _decode(kind, seq_a, seq_b, fn, fd):
    """(sigma [M,1], seg [M,15]|None, rgb [M,32]) exactly as the three decoders compute them (triplane.py:178-270)."""
    if kind == ops.DEC_DISENTANGLED:
        g = _mlp(fn, seq_a)
        return g[:, :1], g[:, 1:], torch.sigmoid(_mlp(fd, seq_b)) * (1 + 2 * 0.001) - 0.001
    x = _mlp(fd, seq_a)
    rgb = torch.sigmoid(x[:, 1:]) * (1 + 2 * 0.001) - 0.001
    return x[:, :1], (_mlp(fd, seq_b) if kind == ops.DEC_SEGMENTATION else None), rgb


def _decoder_params(seq_a, seq_b):
    return [p for seq in (seq_a, seq_b) if seq is not None for p in (seq[0].weight, seq[0].bias, seq[2].weight, seq[2].bias)]


class _FieldBackward:
    """Backward of gather + decoder for one or more passes of samples, accumulated into one set of gradient buffers:
    channel-last plane gradients, decoder-parameter gradients and (single-gather identity) the statistics gradients.
    Samples are either rays x depths (renderer forward) or explicit points (run_model)."""

    def __init__(self, plan, norm_cl, denorm_cl, box_warp, needs_param_grad, dev):
        self.kind, self.seq_a, self.seq_b, self.affine = plan.kind, plan.seq_a, plan.seq_b, plan.affine
        self.norm_cl, self.denorm_cl, self.box_warp, self.dev = norm_cl, denorm_cl, box_warp, dev
        self.params = _decoder_params(plan.seq_a, plan.seq_b)
        self.live = [i for i, need in enumerate(needs_param_grad) if need]
        self.g_params = [torch.zeros_like(p) if i in self.live else None for i, p in enumerate(self.params)]
        any_cl = denorm_cl if denorm_cl is not None else norm_cl
        self.pb, _, self.h, self.w, _ = any_cl.shape
        self.g_denorm_cl = torch.zeros_like(denorm_cl) if denorm_cl is not None else None
        self.g_norm_cl = torch.zeros_like(norm_cl) if norm_cl is not None else None
        self.g_scale = self.g_shift = None
        if self.affine is not None:
            self.g_scale, self.g_shift = torch.zeros_like(self.affine[0]), torch.zeros_like(self.affine[1])
        # one tcgen05 kernel per pass (csrc/nfe_field_bwd.cu, templated on the decoder kind); NFE_BWD_LIBRARY_GEMM=1 keeps the
        # cross-check path: the MLP backward on library GEMMs (torch.addmm) between two gather kernels
        self.fused = not plan.library_gemm
        if self.fused:
            self.full = [g if g is not None else torch.zeros_like(p) for g, p in zip(self.g_params, self.params)]

    def run_pass(self, n, rec, g_rec, rays=None, coords=None):
        """rays = (origins [n,r,3], dirs [n,r,3], depths [n,r,s]) or coords [n,m,3]; rec / g_rec [n*m, 48]."""
        lib, P = _lib.load(), ops._ptr
        stream = torch.cuda.current_stream(self.dev).cuda_stream
        kind, affine = self.kind, self.affine
        if self.fused:
            mlp_a = ops.MlpRef(self.seq_a, self.dev)
            mlp_b = ops.MlpRef(self.seq_b, self.dev) if self.seq_b is not None else None
            grads8 = [P(t) for t in self.full] + [None] * (8 - len(self.full))           # OSG has one net: no second set of parameter gradients
            tail = (mlp_a.ref(), mlp_b.ref() if mlp_b else None, P(rec), P(g_rec), P(self.g_norm_cl), P(self.g_denorm_cl), *grads8,
                    P(affine[0]) if affine else None, P(affine[1]) if affine else None, affine[0].shape[0] if affine else 0,
                    P(self.g_scale), P(self.g_shift), stream)
            if coords is not None:
                _lib.check(lib.nfe_run_model_bwd(kind, P(self.norm_cl), P(self.denorm_cl), self.pb, self.h, self.w, ctypes.c_float(self.box_warp),
                                                 P(coords), n, coords.shape[1], *tail), "nfe_run_model_bwd")
            else:
                o, d, depths = rays
                _lib.check(lib.nfe_field_bwd(kind, P(self.norm_cl), P(self.denorm_cl), self.pb, self.h, self.w, ctypes.c_float(self.box_warp),
                                             P(o), P(d), P(depths), n, o.shape[1], depths.shape[2], *tail), "nfe_field_bwd")
            return
        if coords is not None:
            # explicit points as degenerate rays: origin = point, direction = 0, depth = 0 (o + 0*0 = o exactly)
            o = coords
            d = torch.zeros_like(coords)
            depths = torch.zeros(coords.shape[:2] + (1,), device=self.dev)
        else:
            o, d, depths = rays
        r, s_ = o.shape[1], depths.shape[2]
        total = n * r * s_
        geom = (self.pb, self.h, self.w, ctypes.c_float(self.box_warp), P(o), P(d), P(depths), n, r, s_)
        # decoder inputs
        fd = torch.empty((total, 32), device=self.dev)
        _lib.check(lib.nfe_feature_mean_fwd(P(self.denorm_cl), *geom, P(fd), stream), "nfe_feature_mean_fwd")
        fn = None
        if self.norm_cl is not None:
            fn = torch.empty((total, 32), device=self.dev)
            _lib.check(lib.nfe_feature_mean_fwd(P(self.norm_cl), *geom, P(fn), stream), "nfe_feature_mean_fwd")
        g_flat = g_rec.reshape(total, 48)
        g_fd = torch.empty_like(fd)
        g_fn = torch.empty_like(fn) if fn is not None else None
        # decoder backward on library GEMMs, in row chunks
        for lo in range(0, total, MAX_ROWS):
            hi = min(total, lo + MAX_ROWS)
            with torch.enable_grad():
                xd = fd[lo:hi].detach().requires_grad_(True)
                xn = fn[lo:hi].detach().requires_grad_(True) if fn is not None else None
                sigma, seg, rgb = _decode(kind, self.seq_a, self.seq_b, xn, xd)
                outs, gouts = [sigma, rgb], [g_flat[lo:hi, :1], g_flat[lo:hi, 16:48]]
                if seg is not None:
                    outs.append(seg)
                    gouts.append(g_flat[lo:hi, 1:16])
                inputs = [xd] + ([xn] if xn is not None else []) + [self.params[i] for i in self.live]
                res = torch.autograd.grad(outs, inputs, gouts, allow_unused=True)
            g_fd[lo:hi] = res[0]
            k = 1
            if xn is not None:
                g_fn[lo:hi] = res[1] if res[1] is not None else 0
                k = 2
            for i, g in zip(self.live, res[k:]):
                if g is not None:
                    self.g_params[i] += g
        # gather backward
        _lib.check(lib.nfe_feature_mean_bwd(P(g_fd), *geom, P(self.g_denorm_cl), stream), "nfe_feature_mean_bwd")
        if g_fn is not None:
            _lib.check(lib.nfe_feature_mean_bwd(P(g_fn), *geom, P(self.g_norm_cl), stream), "nfe_feature_mean_bwd")

    def finish(self, norm_shape, plane_shape, need_norm, need_planes, stat_shapes, need_scale, need_shift):
        """(g_norm, g_planes, g_scale, g_shift, g_params) in the reference layouts."""
        lib, P = _lib.load(), ops._ptr
        stream = torch.cuda.current_stream(self.dev).cuda_stream
        if self.fused:
            self.g_params = [self.full[i] if i in self.live else None for i in range(len(self.params))]

        def to_ref(g_cl, shape):
            out = torch.empty(shape, device=self.dev)
            _lib.check(lib.nfe_planes_from_channel_last(P(g_cl), g_cl.shape[0] * 3, 32, self.h * self.w, P(out), stream), "nfe_planes_from_channel_last")
            return out
        g_planes = to_ref(self.g_denorm_cl, plane_shape) if (self.g_denorm_cl is not None and need_planes) else None
        g_norm = to_ref(self.g_norm_cl, norm_shape) if (self.g_norm_cl is not None and need_norm) else None
        g_scale = g_shift = None
        if self.affine is not None:
            g_scale = self.g_scale.reshape(stat_shapes[0]) if need_scale else None
            g_shift = self.g_shift.reshape(stat_shapes[1]) if need_shift else None
        return g_norm, g_planes, g_scale, g_shift, self.g_params


class RenderFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, plan, args, norm_planes, planes, scale_src, shift_src, *params):
        """plan: renderer.field_plan's decision; args: renderer.render_planes' (origins, dirs, depths_coarse, u_fine, opts,
        stochastic, seed, offset).  params are the decoder parameters, passed only so that autograd tracks them; the kernels
        read them from the modules.  scale_src / shift_src: plan.sources or None — under the single-gather identity
        `planes` is never read and its gradient flows through these statistics."""
        cfg, norm_cl, denorm_cl, (rgb, seg, depth, wsum, minmax, st) = render_planes(plan, norm_planes, planes, *args, return_stages=True,
                                                                                      keep_workspace=True)
        ctx.plan, ctx.cfg, ctx.rays = plan, cfg, args[:3]
        ctx.stat_shapes = None if scale_src is None else (scale_src.shape, shift_src.shape)
        ctx.saved = (norm_cl, denorm_cl, st, minmax)
        ctx.plane_shapes = (None if norm_planes is None else norm_planes.shape, planes.shape)
        ctx.mark_non_differentiable(minmax)
        if seg is None:
            return rgb, depth, wsum, minmax
        return rgb, seg, depth, wsum, minmax

    @staticmethod
    def backward(ctx, *grads):
        cfg = ctx.cfg
        norm_cl, denorm_cl, st, minmax = ctx.saved
        if ctx.plan.kind != ops.DEC_OSG:
            g_rgb, g_seg, g_depth, g_wsum = grads[0], grads[1], grads[2], grads[3]
        else:
            g_rgb, g_seg, g_depth, g_wsum = grads[0], None, grads[1], grads[2]
        o, d, depths_coarse = ctx.rays
        n, r, _ = o.shape
        dev = o.device
        s_c, s_f = cfg.s_c, cfg.s_f
        lib = _lib.load()
        stream = torch.cuda.current_stream(dev).cuda_stream

        def f32(t):
            return None if t is None else t.contiguous().float()
        g_rgb = f32(g_rgb) if g_rgb is not None else torch.zeros((n, r, 32), device=dev)
        g_seg, g_depth, g_wsum = f32(g_seg), f32(g_depth), f32(g_wsum)
        dc = depths_coarse.reshape(n, r, s_c).contiguous()
        df = st["depths_fine"].reshape(n, r, s_f).contiguous() if s_f else None
        g_rec_c = torch.empty((n * r, s_c, 48), device=dev)
        g_rec_f = torch.empty((n * r, s_f, 48), device=dev) if s_f else None
        P = ops._ptr
        with torch.cuda.device(dev):
            # 1. compositing backward
            _lib.check(lib.nfe_composite_bwd(P(dc), P(st["sigma_c"]), P(st["rec_c"]), s_c, P(df), P(st.get("sigma_f")), P(st.get("rec_f")), s_f,
                                             n * r, cfg.seg_dim, cfg.white_back, P(g_rgb), P(g_seg), P(g_depth), P(g_wsum), P(minmax),
                                             P(g_rec_c), P(g_rec_f), stream), "nfe_composite_bwd")
            # 2-4. gather + decoder backward of both passes
            fb = _FieldBackward(ctx.plan, norm_cl, denorm_cl, cfg.box_warp, ctx.needs_input_grad[6:], dev)
            for depths, s, rec, g_rec in ((dc, s_c, st["rec_c"], g_rec_c), (df, s_f, st.get("rec_f"), g_rec_f)):
                if s:
                    fb.run_pass(n, rec, g_rec, rays=(o, d, depths))
            # 5. back to the reference layout
            norm_shape, plane_shape = ctx.plane_shapes
            g_norm, g_planes, g_scale, g_shift, g_params = fb.finish(norm_shape, plane_shape, *ctx.needs_input_grad[2:4], ctx.stat_shapes,
                                                                     *ctx.needs_input_grad[4:6])
        return (None, None, g_norm, g_planes, g_scale, g_shift) + tuple(g_params)


class RunModelFunction(torch.autograd.Function):
    """Differentiable run_model (renderer.py:142-148,259-287): the reference's density regulariser back-propagates through
    G.sample_mixed(...)['sigma'] (training/loss.py:310-331, training/triplane.py:150-157).  Gradients reach the plane tensors (or
    the statistics, under the single-gather identity) and the decoder parameters; the sample coordinates carry none."""

    @staticmethod
    def forward(ctx, plan, args, norm_planes, planes, scale_src, shift_src, *params):
        """As RenderFunction.forward; args: renderer.run_model_planes' (coords, opts, seed, offset, sigma_only)."""
        cfg, norm_cl, denorm_cl, out = run_model_planes(plan, norm_planes, planes, *args)
        ctx.plan, ctx.coords, ctx.box_warp = plan, args[0], cfg.box_warp
        ctx.stat_shapes = None if scale_src is None else (scale_src.shape, shift_src.shape)
        ctx.saved = (norm_cl, denorm_cl, out.get("rgb"))
        ctx.plane_shapes = (None if norm_planes is None else norm_planes.shape, planes.shape)
        ctx.keys = tuple(k for k in ("rgb", "sigma", "seg") if k in out)
        return tuple(out[k] for k in ctx.keys)

    @staticmethod
    def backward(ctx, *grads):
        coords = ctx.coords
        norm_cl, denorm_cl, rgb = ctx.saved
        n, m, _ = coords.shape
        dev = coords.device
        g = dict(zip(ctx.keys, grads))
        # records {sigma, seg[15], rgb[32]} of the forward (only the colours are read: sigmoid derivative) and of the gradients
        rec = torch.zeros((n * m, 48), device=dev)
        g_rec = torch.zeros((n * m, 48), device=dev)
        if rgb is not None:
            rec[:, 16:48] = rgb.reshape(n * m, 32)
        if g.get("sigma") is not None:
            g_rec[:, 0:1] = g["sigma"].reshape(n * m, 1)
        if g.get("seg") is not None:
            g_rec[:, 1:16] = g["seg"].reshape(n * m, 15)
        if g.get("rgb") is not None:
            g_rec[:, 16:48] = g["rgb"].reshape(n * m, 32)
        with torch.cuda.device(dev):
            fb = _FieldBackward(ctx.plan, norm_cl, denorm_cl, ctx.box_warp, ctx.needs_input_grad[6:], dev)
            fb.run_pass(n, rec, g_rec, coords=coords)
            norm_shape, plane_shape = ctx.plane_shapes
            g_norm, g_planes, g_scale, g_shift, g_params = fb.finish(norm_shape, plane_shape, *ctx.needs_input_grad[2:4], ctx.stat_shapes,
                                                                     *ctx.needs_input_grad[4:6])
        return (None, None, g_norm, g_planes, g_scale, g_shift) + tuple(g_params)


class NormalizeFunction(torch.autograd.Function):
    """normalize_plane with its analytic backward (triplane.py:56-65): n = (x - mean) / (std + 1e-8).
    Returns (norm, mean, std, norm_cl): norm_cl is the channel-last staging written by the same kernel (None for tensors
    that are not [N,96,H,W] tri-planes); triplane.normalize_plane registers it against the tensors the caller sees."""

    @staticmethod
    def forward(ctx, planes):
        mean, std = ops.plane_stats(planes)
        norm_cl = None
        if planes.dim() == 4 and planes.shape[1] == 96 and planes.is_contiguous() and planes.dtype == torch.float32:
            # the raw set is staged on demand (single-gather identity: never)
            norm, norm_cl, _ = ops.plane_normalize_staged(planes.detach(), mean, std, register=False)
        else:
            norm = ops.plane_normalize(planes, mean, std)
        ctx.save_for_backward(norm, std)
        ctx.hw = planes.shape[-1] * planes.shape[-2]
        if norm_cl is None:
            return norm, mean, std, None
        ctx.mark_non_differentiable(norm_cl)
        return norm, mean, std, norm_cl

    @staticmethod
    def backward(ctx, g_norm, g_mean, g_std, _g_cl=None):
        norm, std = ctx.saved_tensors
        # d n_j / d x_i = (delta_ij - 1/N)/d - n_j * n_i * d / ((N-1) * std * d)   (std is the unbiased one), i.e.
        #   gx = (g - mean(g))/d - norm*sum(g*norm)/((N-1)*std) + g_mean/N + g_std*norm*d/((N-1)*std)
        # in two streaming CUDA passes (csrc/nfe_planes.cu)
        def f32(t):
            return None if t is None else t.contiguous().float()
        g, gm, gs = f32(g_norm), f32(g_mean), f32(g_std)
        slabs = norm.numel() // ctx.hw
        gx = torch.empty_like(norm)
        sums = torch.empty((slabs, 2), device=norm.device, dtype=torch.float64) if g is not None else None
        with torch.cuda.device(norm.device):
            _lib.check(_lib.load().nfe_plane_normalize_bwd(ops._ptr(g), ops._ptr(norm), ops._ptr(std), ops._ptr(gm), ops._ptr(gs), slabs, ctx.hw,
                                                           ops._ptr(sums), ops._ptr(gx), torch.cuda.current_stream(norm.device).cuda_stream),
                       "nfe_plane_normalize_bwd")
        return gx


class DenormalizeFunction(torch.autograd.Function):
    """denormalize_plane (triplane.py:66-68): out = planes * std + mean, statistics broadcast over H, W (and over the
    batch when they belong to a single item)."""

    @staticmethod
    def forward(ctx, planes, mean, std):
        ctx.save_for_backward(planes, std)
        ctx.stat_shape = mean.shape
        return ops.plane_denormalize(planes, mean, std, register=False)

    @staticmethod
    def backward(ctx, g):
        planes, std = ctx.saved_tensors

        def reduce_to(t, shape):
            t = t.sum(dim=(-1, -2), keepdim=True)
            if shape[0] == 1 and t.shape[0] != 1:
                t = t.sum(dim=0, keepdim=True)
            return t.reshape(shape)
        return (g * std if ctx.needs_input_grad[0] else None,
                reduce_to(g, ctx.stat_shape) if ctx.needs_input_grad[1] else None,
                reduce_to(g * planes, ctx.stat_shape) if ctx.needs_input_grad[2] else None)
