"""A plain-torch restatement of the reference's differentiable render path, in any floating dtype, differentiable by autograd.

It restates training/volumetric_rendering/renderer.py:39-65,150-167,288-300 (tri-plane gather, merge of the two passes),
ray_marcher.py:25-57,68-101 (MipRayMarcher2 / SegMipRayMarcher2) and training/triplane.py:167-270 (the three decoders with
FullyConnectedLayer gains).  It is the independent side of the backward parity tests: run in float64 it gives the gradient
the CUDA backward is compared with.  Sampling is not restated.  The coarse and fine depths are inputs, as the reference
detaches the fine depths (renderer.py:198,211), so the gradient does not depend on how they were drawn.

It reads the decoder parameters from the package's decoder modules as plain tensors and imports nothing else of the package.
"""
import torch
import torch.nn.functional as F


def sample_from_planes(planes, coords, box_warp):
    """planes [N|1,3,C,H,W], coords [N,M,3] -> [N,3,M,C] (renderer.py:39-65): scale by 2/box_warp, project onto
    (x,y), (x,z), (z,x), bilinear grid_sample with zero padding and align_corners=False.  A batch-1 plane set is
    expanded over the N coordinate sets."""
    n, m, _ = coords.shape
    if planes.shape[0] == 1 and n > 1:
        planes = planes.expand(n, *planes.shape[1:])
    _, n_planes, c, h, w = planes.shape
    q = (2 / box_warp) * coords
    grid = torch.stack([q[..., [0, 1]], q[..., [0, 2]], q[..., [2, 0]]], dim=1)          # [N,3,M,2]
    out = F.grid_sample(planes.reshape(n * n_planes, c, h, w), grid.reshape(n * n_planes, 1, m, 2), mode='bilinear',
                        padding_mode='zeros', align_corners=False)
    return out.permute(0, 3, 2, 1).reshape(n, n_planes, m, c)


class Decoder:
    """One of the three decoders (triplane.py:167-270) over leaf copies of a decoder module's parameters.

    `params` maps the module's parameter names ('net.0.weight', 'geo_net.2.bias', ...) to leaf tensors of `dtype` that
    require grad, so `params[name].grad` is the gradient autograd takes through this restatement."""

    def __init__(self, module, dtype=torch.float64, device=None):
        if hasattr(module, "geo_net"):
            self.kind, self.nets = "dis", ("geo_net", "app_net")
        elif hasattr(module, "seg_net"):
            self.kind, self.nets = "seg", ("net", "seg_net")
        else:
            self.kind, self.nets = "osg", ("net",)
        self.params = {name: p.detach().to(device=device, dtype=dtype).clone().requires_grad_(True)
                       for name, p in module.named_parameters()}
        self.gains = {net: tuple(float(g) for g in (getattr(module, net)[0].weight_gain, getattr(module, net)[0].bias_gain,
                                                    getattr(module, net)[2].weight_gain, getattr(module, net)[2].bias_gain))
                      for net in self.nets}

    def _fc(self, x, net, i, weight_gain, bias_gain):
        """FullyConnectedLayer, activation='linear' (networks_stylegan2.py:114-123)."""
        w = self.params[f"{net}.{i}.weight"] * weight_gain
        b = self.params[f"{net}.{i}.bias"]
        if bias_gain != 1:
            b = b * bias_gain
        return torch.addmm(b.unsqueeze(0), x, w.t())

    def _mlp(self, x, net):
        wg1, bg1, wg2, bg2 = self.gains[net]
        return self._fc(F.softplus(self._fc(x, net, 0, wg1, bg1)), net, 2, wg2, bg2)

    def __call__(self, sampled_norm, sampled_denorm):
        """[N,3,M,C] features (sampled_norm is unused by OSG and Segmentation) -> dict(rgb, sigma[, seg]) of [N,M,*]."""
        n, _, m, c = sampled_denorm.shape
        fd = sampled_denorm.mean(1).reshape(n * m, c)
        if self.kind == "dis":
            g = self._mlp(sampled_norm.mean(1).reshape(n * m, c), "geo_net")
            rgb = torch.sigmoid(self._mlp(fd, "app_net")) * (1 + 2 * 0.001) - 0.001
            out = {"rgb": rgb, "sigma": g[:, 0:1], "seg": g[:, 1:]}
        else:
            x = self._mlp(fd, "net")
            out = {"rgb": torch.sigmoid(x[:, 1:]) * (1 + 2 * 0.001) - 0.001, "sigma": x[:, 0:1]}
            if self.kind == "seg":
                out["seg"] = self._mlp(fd, "seg_net")
        return {k: v.reshape(n, m, v.shape[-1]) for k, v in out.items()}


def run_model(decoder, norm_planes, planes, coords, box_warp):
    """renderer.py:142-148,259-287 without density noise: gather and decode at explicit points."""
    fd = sample_from_planes(planes, coords, box_warp)
    fn = sample_from_planes(norm_planes, coords, box_warp) if decoder.kind == "dis" else None
    return decoder(fn, fd)


def march(colors, densities, depths, segs=None, white_back=False):
    """MipRayMarcher2 / SegMipRayMarcher2 (ray_marcher.py:25-57,68-101).  [N,R,S,*] -> (rgb, seg|None, depth, weights).

    One deviation, in the backward only: where the weight total is exactly 0 the reference's depth is 0/0 = NaN, which
    nan_to_num and the clamp turn into the global maximum depth, and whose autograd gradient is NaN (division backward of
    0/0).  Here that division is taken with a denominator of 1 and the NaN put back by torch.where, so the forward is the
    reference's and the gradient through the depth of such a ray is 0, the value the kernels define."""
    deltas = depths[:, :, 1:] - depths[:, :, :-1]
    colors_mid = (colors[:, :, :-1] + colors[:, :, 1:]) / 2
    densities_mid = (densities[:, :, :-1] + densities[:, :, 1:]) / 2
    depths_mid = (depths[:, :, :-1] + depths[:, :, 1:]) / 2
    densities_mid = F.softplus(densities_mid - 1)
    alpha = 1 - torch.exp(-(densities_mid * deltas))
    alpha_shifted = torch.cat([torch.ones_like(alpha[:, :, :1]), 1 - alpha + 1e-10], -2)
    weights = alpha * torch.cumprod(alpha_shifted, -2)[:, :, :-1]
    composite_rgb = torch.sum(weights * colors_mid, -2)
    composite_seg = None
    if segs is not None:
        segs_mid = (segs[:, :, :-1] + segs[:, :, 1:]) / 2
        composite_seg = torch.sum(weights * segs_mid, -2)
    weight_total = weights.sum(2)
    empty = weight_total == 0
    composite_depth = torch.sum(weights * depths_mid, -2) / torch.where(empty, torch.ones_like(weight_total), weight_total)
    composite_depth = torch.where(empty, torch.full_like(composite_depth, float('nan')), composite_depth)
    composite_depth = torch.nan_to_num(composite_depth, float('inf'))
    composite_depth = torch.clamp(composite_depth, torch.min(depths), torch.max(depths))
    if white_back:
        composite_rgb = composite_rgb + 1 - weight_total
    composite_rgb = composite_rgb * 2 - 1
    return composite_rgb, composite_seg, composite_depth, weights


def unify(depths_coarse, depths_fine, attrs_coarse, attrs_fine):
    """Concatenate the two passes and sort by depth (renderer.py:157-167,288-300), stably: on exact ties the order
    differs from an unstable sort only in which of two samples at the same position comes first."""
    all_depths = torch.cat([depths_coarse, depths_fine], dim=-2)
    _, indices = torch.sort(all_depths, dim=-2, stable=True)
    out = {k: torch.gather(torch.cat([attrs_coarse[k], attrs_fine[k]], dim=-2), -2, indices.expand(-1, -1, -1, attrs_coarse[k].shape[-1]))
           for k in attrs_coarse}
    return torch.gather(all_depths, -2, indices), out


def _evaluate(decoder, norm_planes, planes, origins, dirs, depths, box_warp):
    n, r, s, _ = depths.shape
    coords = (origins.unsqueeze(-2) + depths * dirs.unsqueeze(-2)).reshape(n, -1, 3)
    out = run_model(decoder, norm_planes, planes, coords, box_warp)
    return {k: v.reshape(n, r, s, v.shape[-1]) for k, v in out.items()}


def render(decoder, norm_planes, planes, origins, dirs, depths_coarse, depths_fine, box_warp=1.0, white_back=False):
    """renderer.py:88-140,301-363 from given depths: depths_coarse [N,R,S_c(,1)], depths_fine [N,R,S_f(,1)] or None for a
    single pass.  Rays and depths are cast to the planes' dtype.  Returns (rgb [N,R,32], seg [N,R,15]|None, depth [N,R,1],
    weights.sum(2) [N,R,1])."""
    dt = planes.dtype

    def as_samples(d):
        d = d.to(dt)
        return d if d.dim() == 4 else d.unsqueeze(-1)
    origins, dirs = origins.to(dt), dirs.to(dt)
    depths = as_samples(depths_coarse)
    out = _evaluate(decoder, norm_planes, planes, origins, dirs, depths, box_warp)
    if depths_fine is not None:
        fine = as_samples(depths_fine)
        depths, out = unify(depths, fine, out, _evaluate(decoder, norm_planes, planes, origins, dirs, fine, box_warp))
    rgb, seg, depth, weights = march(out["rgb"], out["sigma"], depths, out.get("seg"), white_back)
    return rgb, seg, depth, weights.sum(2)
