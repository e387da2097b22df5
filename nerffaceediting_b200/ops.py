"""Tensor-level wrappers over the C ABI: torch supplies device memory and the stream, nothing else.

Each function validates like the reference's plugins do with TORCH_CHECK (torch_utils/ops/bias_act.cpp:39-55):
wrong device / dtype raises RuntimeError; there is no CPU path.
"""
import ctypes

import os

import torch

from . import _lib
from . import plane_registry as registry
from ._lib import DEC_DISENTANGLED, DEC_OSG, DEC_SEGMENTATION, NfeMlp, NfeRenderCfg  # noqa: F401


def _cuda_f32(t, name):
    if not isinstance(t, torch.Tensor):
        raise RuntimeError(f"{name}: expected a tensor, got {type(t).__name__}")
    if not t.is_cuda:
        raise RuntimeError(f"{name}: expected a CUDA tensor (this path has no CPU fallback), got device {t.device}")
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


def _ptr(t):
    return None if t is None else t.data_ptr()


def _stream(t):
    return torch.cuda.current_stream(t.device).cuda_stream


class _Guard:
    """Current-device guard (the reference plugins use OptionalCUDAGuard, bias_act.cpp:58)."""

    def __init__(self, t):
        self.ctx = torch.cuda.device(t.device)

    def __enter__(self):
        self.ctx.__enter__()

    def __exit__(self, *a):
        self.ctx.__exit__(*a)


def _no_grad_needed(*tensors):
    if torch.is_grad_enabled() and any(isinstance(t, torch.Tensor) and t.requires_grad for t in tensors):
        raise RuntimeError("nerffaceediting_b200: the backward pass of this op is not built yet; "
                           "call under torch.no_grad() or detach the inputs")


# ------------------------------------------------------------------------------- plane statistics
def plane_stats(planes):
    """mean / std (sqrt of unbiased variance) over the last two dims, keepdim (triplane.py:56-60)."""
    x = _cuda_f32(planes, "planes")
    hw = x.shape[-1] * x.shape[-2]
    slabs = x.numel() // max(hw, 1)
    mean = torch.empty(x.shape[:-2] + (1, 1), device=x.device, dtype=torch.float32)
    std = torch.empty_like(mean)
    with _Guard(x):
        _lib.check(_lib.load().nfe_plane_stats(_ptr(x), slabs, hw, _ptr(mean), _ptr(std), _stream(x)), "nfe_plane_stats")
    return mean, std


def plane_normalize(planes, mean, std):
    x = _cuda_f32(planes, "planes")
    mean, std = _cuda_f32(mean, "mean"), _cuda_f32(std, "std")
    hw = x.shape[-1] * x.shape[-2]
    slabs = x.numel() // max(hw, 1)
    if mean.numel() != slabs or std.numel() != slabs:
        raise RuntimeError("plane_normalize: statistics do not match the planes")
    out = torch.empty_like(x)
    with _Guard(x):
        _lib.check(_lib.load().nfe_plane_normalize(_ptr(x), _ptr(mean), _ptr(std), slabs, hw, _ptr(out), _stream(x)), "nfe_plane_normalize")
    return out


def plane_denormalize(norm, mean, std, register=True):
    """norm*std + mean; statistics either per (batch, channel) or one item's, broadcast over the batch."""
    x = _cuda_f32(norm, "planes")
    hw = x.shape[-1] * x.shape[-2]
    slabs = x.numel() // max(hw, 1)
    mean = _cuda_f32(torch.as_tensor(mean, device=x.device), "mean")
    std = _cuda_f32(torch.as_tensor(std, device=x.device), "std")
    if mean.numel() != std.numel():
        mean, std = torch.broadcast_tensors(mean, std)
        mean, std = mean.contiguous(), std.contiguous()
    stat = mean.numel()
    per_item = slabs // max(x.shape[0], 1)
    if stat not in (slabs, per_item):
        # arbitrary broadcast (rare): expand to one entry per slab
        mean = mean.expand(x.shape[:-2] + (1, 1)).contiguous()
        std = std.expand(x.shape[:-2] + (1, 1)).contiguous()
        stat = slabs
    out = torch.empty_like(x)
    with _Guard(x):
        _lib.check(_lib.load().nfe_plane_denormalize(_ptr(x), _ptr(mean), _ptr(std), slabs, stat, hw, _ptr(out), _stream(x)),
                   "nfe_plane_denormalize")
    if register and x is norm:         # (a converted temporary cannot be identified later)
        register_denormalized(out, norm, mean, std)
    return out


def register_denormalized(out, norm, mean, std):
    """Record out == norm*std + mean per (item, plane-major channel) when the statistics have that form (tri-plane tensors
    with one statistics row per item, or one row for the whole batch): the single-gather identity then also holds after a
    statistics swap (triplane.py:93-107)."""
    if not (torch.is_tensor(mean) and torch.is_tensor(std)) or mean.numel() != std.numel():
        return
    if norm.dim() in (4, 5) and (norm.shape[1] == 96 or (norm.dim() == 5 and norm.shape[1] == 3 and norm.shape[2] == 32)):
        stat = mean.numel()
        k = stat // 96 if stat % 96 == 0 else 0
        if k in (1, norm.shape[0]):
            registry.provenance_put(out, norm, std.detach().reshape(k, 96).float(), mean.detach().reshape(k, 96).float())


def resize_bilinear(x, size, antialias=True):
    """torch.nn.functional.interpolate(x, size=(size, size), mode='bilinear', align_corners=False, antialias=antialias)
    for the super-resolution module's input (superresolution.py:48-52,80-84,282-286; SURVEY.md §8f f1).  x [N,C,H,W]."""
    x = _cuda_f32(x, "x")
    if x.dim() != 4:
        raise RuntimeError(f"resize_bilinear: expected [N,C,H,W], got {tuple(x.shape)}")
    _no_grad_needed(x)
    n, c, h, w = x.shape
    oh, ow = (int(size), int(size)) if isinstance(size, int) else (int(size[0]), int(size[1]))
    out = torch.empty((n, c, oh, ow), device=x.device, dtype=torch.float32)
    with _Guard(x):
        _lib.check(_lib.load().nfe_resize_bilinear(_ptr(x), n * c, h, w, oh, ow, int(bool(antialias)), _ptr(out), _stream(x)), "nfe_resize_bilinear")
    return out


# Registries (plane_registry.py): staged channel-last copies and the provenance of de-normalised planes
_key5 = registry.key5
_version_of = registry.version_of
provenance = registry.provenance
provenance_attach = registry.provenance_attach
provenance_sources = registry.provenance_sources
note_path = registry.note
path_counts = registry.counts


def planes_channel_last(planes, cache=False):
    """[N,3,C,H,W] (reference layout) -> channel-last [N,3,H,W,C] staging buffer for the gather.
    With cache=True (rendering_options['nfe_cache_planes']) the staged copy is kept, keyed on
    (address, shape, version) and valid while the source tensor is alive, so a video sweep over fixed planes
    (utils.py:78-80) stages once."""
    x = _cuda_f32(planes, "planes")
    if x.dim() != 5 or x.shape[1] != 3:
        raise RuntimeError(f"planes: expected [N,3,C,H,W], got {tuple(x.shape)}")
    hit = registry.staged_get(x)      # staged by normalize_plane, or kept from an earlier call with cache=True
    if hit is not None:
        return hit
    n, p, c, h, w = x.shape
    out = torch.empty((n, p, h, w, c), device=x.device, dtype=torch.float32)
    with _Guard(x):
        _lib.check(_lib.load().nfe_planes_to_channel_last(_ptr(x), n * p, c, h * w, _ptr(out), _stream(x)), "nfe_planes_to_channel_last")
    if cache and x is planes:         # (a converted temporary would die at once and take the entry with it)
        registry.staged_put(planes, out)
    return out


def plane_normalize_staged(planes, mean, std, stage_raw=False, register=True):
    """normalize_plane for tri-plane tensors [N, 96, H, W]: one kernel writes the normalised planes AND the
    channel-last staging of both the normalised and the raw planes.  Returns (norm, norm_cl, raw_cl|None).
    register=True also records the staged copies and the provenance (raw == norm*(std+1e-8) + mean) so that the
    renderer called next on views of (norm, planes) (triplane.py:113-119) skips its own staging pass and gathers
    one plane set; the entries live as long as `planes` and the returned `norm` do."""
    x = _cuda_f32(planes, "planes")
    n, c96, h, w = x.shape
    norm = torch.empty_like(x)
    norm_cl = torch.empty((n, 3, h, w, 32), device=x.device, dtype=torch.float32)
    raw_cl = torch.empty_like(norm_cl) if stage_raw else None
    with _Guard(x):
        _lib.check(_lib.load().nfe_plane_normalize_staged(_ptr(x), _ptr(mean), _ptr(std), n * 3, h * w, _ptr(norm), _ptr(norm_cl), _ptr(raw_cl),
                                                          _stream(x)), "nfe_plane_normalize_staged")
    if register:
        register_normalized(planes, norm, mean, std, norm_cl, raw_cl)
    return norm, norm_cl, raw_cl


def register_normalized(planes, norm, mean, std, norm_cl, raw_cl=None):
    """Record what normalize_plane knows about its input and output: the staged copies, and that the raw planes ARE the
    de-normalisation of `norm` with their own statistics."""
    n = planes.shape[0]
    registry.staged_put(norm, norm_cl)
    if raw_cl is not None:
        registry.staged_put(planes, raw_cl)
    registry.provenance_put(planes, norm, std.detach().reshape(n, -1) + 1e-8, mean.detach().reshape(n, -1))


def clear_plane_cache():
    """Drop every staged copy and provenance record (and the autograd sources attached to them)."""
    registry.clear()


# ------------------------------------------------------------------------------- rays
def generate_rays(cam2world, intrinsics, resolution):
    c = _cuda_f32(cam2world, "cam2world_matrix").reshape(-1, 16)
    k = _cuda_f32(intrinsics, "intrinsics").reshape(-1, 9)
    if c.shape[0] != k.shape[0]:
        raise RuntimeError("generate_rays: cam2world and intrinsics batch sizes differ")
    n, res = c.shape[0], int(resolution)
    o = torch.empty((n, res * res, 3), device=c.device, dtype=torch.float32)
    d = torch.empty_like(o)
    with _Guard(c):
        _lib.check(_lib.load().nfe_generate_rays(_ptr(c), _ptr(k), n, res, _ptr(o), _ptr(d), _stream(c)), "nfe_generate_rays")
    return o, d


def ray_limits_box(origins, dirs, box_side_length):
    o, d = _cuda_f32(origins, "rays_o"), _cuda_f32(dirs, "rays_d")
    tmin = torch.empty(o.shape[:-1] + (1,), device=o.device, dtype=torch.float32)
    tmax = torch.empty_like(tmin)
    with _Guard(o):
        _lib.check(_lib.load().nfe_ray_limits_box(_ptr(o), _ptr(d), o.numel() // 3, float(box_side_length), _ptr(tmin), _ptr(tmax), _stream(o)),
                   "nfe_ray_limits_box")
    return tmin, tmax


_TABLES = {}


def linspace_table(start, end, steps, device):
    """torch.linspace evaluated on the HOST and uploaded: its fp32 values are not reproducible by
    start + i*step (SURVEY.md §7.5), and the CPU reference is the oracle."""
    key = (float(start), float(end), int(steps), str(device))
    t = _TABLES.get(key)
    if t is None:
        t = torch.linspace(start, end, steps).to(device)
        if len(_TABLES) > 64:
            _TABLES.clear()
        _TABLES[key] = t
    return t


_PHILOX_DRAWS = [0]


def philox_draws():
    """How many times a call asked for a Philox (seed, offset) so far; graphs.capture uses it to refuse calls whose random
    state would be frozen into a CUDA graph."""
    return _PHILOX_DRAWS[0]


def philox_state(device, n_streams=4):
    """(seed, offset) from torch's CUDA generator, advanced so successive calls differ and
    torch.manual_seed makes stochastic renders reproducible."""
    _PHILOX_DRAWS[0] += 1
    gen = torch.cuda.default_generators[device.index if device.index is not None else torch.cuda.current_device()]
    seed, offset = gen.initial_seed(), gen.get_offset()
    gen.set_offset(offset + 4 * n_streams)
    return seed & 0xFFFFFFFFFFFFFFFF, offset


def sample_stratified(n, r, s_c, device, ray_start, ray_end, disparity=False, jitter=None, stochastic=False, seed=0, offset=0):
    """depths_coarse [N,R,S,1] (renderer.py:169-192).  ray_start/ray_end: floats, or [N,R,1] tensors."""
    out = torch.empty((n, r, s_c, 1), device=device, dtype=torch.float32)
    lib = _lib.load()
    jit = _cuda_f32(jitter, "jitter") if jitter is not None else None
    with torch.cuda.device(device):
        stream = torch.cuda.current_stream(device).cuda_stream
        if disparity:
            table = linspace_table(0, 1, s_c, device)
            rc = lib.nfe_sample_stratified(n * r, s_c, 2, _ptr(table), float(ray_start), float(ray_end), None, None, _ptr(jit),
                                           int(stochastic), seed, offset, _ptr(out), stream)
        elif isinstance(ray_start, torch.Tensor):
            a, b = _cuda_f32(ray_start, "ray_start"), _cuda_f32(ray_end, "ray_end")
            rc = lib.nfe_sample_stratified(n * r, s_c, 1, None, 0.0, 0.0, _ptr(a), _ptr(b), _ptr(jit), int(stochastic), seed, offset,
                                           _ptr(out), stream)
        else:
            table = linspace_table(ray_start, ray_end, s_c, device)
            rc = lib.nfe_sample_stratified(n * r, s_c, 0, _ptr(table), float(ray_start), float(ray_end), None, None, _ptr(jit),
                                           int(stochastic), seed, offset, _ptr(out), stream)
    _lib.check(rc, "nfe_sample_stratified")
    return out


# ------------------------------------------------------------------------------- gather / decoders
def sample_planes(planes_cl, coords, box_warp):
    """planes_cl [Np,3,H,W,C] channel-last, coords [N,M,3] -> [N,3,M,C]."""
    co = _cuda_f32(coords, "coordinates")
    np_, _, h, w, c = planes_cl.shape
    n, m, _ = co.shape
    out = torch.empty((n, 3, m, c), device=co.device, dtype=torch.float32)
    with _Guard(co):
        _lib.check(_lib.load().nfe_sample_planes_fwd(_ptr(planes_cl), np_, c, h, w, _ptr(co), n, m, float(box_warp), _ptr(out), _stream(co)),
                   "nfe_sample_planes_fwd")
    return out


def _fc_ok(layer):
    return (hasattr(layer, "weight") and getattr(layer, "bias", None) is not None and hasattr(layer, "weight_gain")
            and hasattr(layer, "bias_gain") and getattr(layer, "activation", "linear") == "linear" and layer.weight.dim() == 2)


def _mlp_ok(seq):
    try:
        if len(seq) != 3 or not _fc_ok(seq[0]) or not _fc_ok(seq[2]):
            return False
        act = seq[1]
        return (type(act).__name__ == "Softplus" and float(getattr(act, "beta", 1)) == 1.0
                and float(getattr(act, "threshold", 20)) == 20.0 and seq[0].weight.shape[0] == seq[2].weight.shape[1])
    except TypeError:
        return False


def describe_decoder(decoder):
    """Recognise the reference's decoders BY STRUCTURE (SURVEY.md §7.9: persistent classes make isinstance
    unreliable): geo_net+app_net -> Disentangled, net+seg_net -> Segmentation, net -> OSG, each a
    Sequential(FC, Softplus, FC) with 32->64->{16,32,33,15}.  Returns (kind, seq_a, seq_b) or None."""
    def dims(seq):
        return (seq[0].weight.shape[1], seq[0].weight.shape[0], seq[2].weight.shape[0])
    geo, app = getattr(decoder, "geo_net", None), getattr(decoder, "app_net", None)
    net, seg = getattr(decoder, "net", None), getattr(decoder, "seg_net", None)
    if geo is not None and app is not None and _mlp_ok(geo) and _mlp_ok(app):
        if dims(geo) == (32, 64, 16) and dims(app) == (32, 64, 32):
            return DEC_DISENTANGLED, geo, app
        return None
    if net is not None and seg is not None and _mlp_ok(net) and _mlp_ok(seg):
        if dims(net) == (32, 64, 33) and dims(seg) == (32, 64, 15):
            return DEC_SEGMENTATION, net, seg
        return None
    if net is not None and geo is None and seg is None and _mlp_ok(net) and dims(net) == (32, 64, 33):
        return DEC_OSG, net, None
    return None


class MlpRef:
    """nfe_mlp view of a Sequential(FC, Softplus, FC); keeps the fp32 contiguous tensors alive."""

    def __init__(self, seq, device):
        a, b = seq[0], seq[2]
        self.keep = [_cuda_f32(a.weight.detach().to(device), "weight"), _cuda_f32(a.bias.detach().to(device), "bias"),
                     _cuda_f32(b.weight.detach().to(device), "weight"), _cuda_f32(b.bias.detach().to(device), "bias")]
        self.c = NfeMlp(self.keep[0].data_ptr(), self.keep[1].data_ptr(), self.keep[2].data_ptr(), self.keep[3].data_ptr(),
                        a.weight.shape[1], a.weight.shape[0], b.weight.shape[0],
                        float(a.weight_gain), float(a.bias_gain), float(b.weight_gain), float(b.bias_gain))

    def ref(self):
        return ctypes.byref(self.c)


def decoder_fwd(kind, seq_a, seq_b, feat_norm, feat_denorm, precision=_lib.PREC_FP32):
    """decoder(sampled_features [N,3,M,32]...) -> dict(rgb [N,M,32], sigma [N,M,1][, seg [N,M,15]])."""
    fd = _cuda_f32(feat_denorm, "sampled_features")
    fn = _cuda_f32(feat_norm, "sampled_norm_features") if (feat_norm is not None and kind == DEC_DISENTANGLED) else None
    if fd.dim() != 4 or fd.shape[1] != 3:
        raise RuntimeError(f"sampled_features: expected [N,3,M,C], got {tuple(fd.shape)}")
    n, _, m, c = fd.shape
    a = MlpRef(seq_a, fd.device)
    b = MlpRef(seq_b, fd.device) if seq_b is not None else None
    rgb = torch.empty((n, m, 32), device=fd.device, dtype=torch.float32)
    sigma = torch.empty((n, m, 1), device=fd.device, dtype=torch.float32)
    seg = torch.empty((n, m, 15), device=fd.device, dtype=torch.float32) if kind != DEC_OSG else None
    with _Guard(fd):
        _lib.check(_lib.load().nfe_decoder_fwd(kind, int(precision), a.ref(), b.ref() if b else None, _ptr(fn), _ptr(fd), n, m, c, _ptr(rgb), _ptr(sigma),
                                               _ptr(seg), _stream(fd)), "nfe_decoder_fwd")
    out = {"rgb": rgb, "sigma": sigma}
    if seg is not None:
        out["seg"] = seg
    return out


# ------------------------------------------------------------------------------- marching
def composite(colors, sigma, depths, segs=None, white_back=False):
    """[N,R,S,*] -> rgb [N,R,cc], seg [N,R,cs]|None, depth [N,R,1], weights [N,R,S-1,1]."""
    col, sg, dp = _cuda_f32(colors, "colors"), _cuda_f32(sigma, "densities"), _cuda_f32(depths, "depths")
    n, r, s, cc = col.shape
    sgs = _cuda_f32(segs, "segs") if segs is not None else None
    cs = sgs.shape[-1] if sgs is not None else 0
    dev = col.device
    rgb = torch.empty((n, r, cc), device=dev, dtype=torch.float32)
    seg = torch.empty((n, r, cs), device=dev, dtype=torch.float32) if cs else None
    depth = torch.empty((n, r, 1), device=dev, dtype=torch.float32)
    weights = torch.empty((n, r, s - 1, 1), device=dev, dtype=torch.float32)
    mm = torch.empty(2, device=dev, dtype=torch.float32)
    with _Guard(col):
        _lib.check(_lib.load().nfe_composite_fwd(_ptr(col), _ptr(sgs), _ptr(sg), _ptr(dp), n * r, s, cc, cs, int(bool(white_back)),
                                                 _ptr(rgb), _ptr(seg), _ptr(depth), _ptr(weights), None, _ptr(mm), _stream(col)),
                   "nfe_composite_fwd")
    return rgb, seg, depth, weights


def importance_resample(z_vals, weights, s_f, u=None, seed=0, offset=0, return_indices=False):
    """z_vals [Rn,S], weights [Rn,S-1] -> [Rn,S_f]; u None -> Philox U[0,1) (sample_pdf det=False)."""
    z, w = _cuda_f32(z_vals, "z_vals"), _cuda_f32(weights, "weights")
    rn, s = z.shape
    if w.shape != (rn, s - 1):
        raise RuntimeError(f"importance_resample: weights must be [{rn},{s - 1}], got {tuple(w.shape)}")
    uu = _cuda_f32(u, "u") if u is not None else None
    out = torch.empty((rn, s_f), device=z.device, dtype=torch.float32)
    below = torch.empty((rn, s_f), device=z.device, dtype=torch.int32) if return_indices else None
    above = torch.empty_like(below) if return_indices else None
    with _Guard(z):
        _lib.check(_lib.load().nfe_importance_resample(_ptr(z), _ptr(w), rn, s, int(s_f), _ptr(uu), int(uu is not None and uu.dim() == 2),
                                                       seed, offset, _ptr(out), _ptr(below), _ptr(above), _stream(z)),
                   "nfe_importance_resample")
    return (out, below, above) if return_indices else out


def sample_pdf(bins, weights, s_f, u=None, seed=0, offset=0, eps=1e-5):
    """sample_pdf(bins [Rn,nb], weights [Rn,ns]) -> [Rn,S_f]   (renderer.py:214-253)."""
    b, w = _cuda_f32(bins, "bins"), _cuda_f32(weights, "weights")
    rn, nb = b.shape
    ns = w.shape[1]
    uu = _cuda_f32(u, "u") if u is not None else None
    out = torch.empty((rn, s_f), device=b.device, dtype=torch.float32)
    with _Guard(b):
        _lib.check(_lib.load().nfe_sample_pdf(_ptr(b), _ptr(w), rn, nb, ns, int(s_f), _ptr(uu), int(uu is not None and uu.dim() == 2),
                                              seed, offset, float(eps), _ptr(out), _stream(b)), "nfe_sample_pdf")
    return out


def unify_samples(depths1, colors1, sigma1, depths2, colors2, sigma2, segs1=None, segs2=None):
    """cat + sort by depth + gather of every attribute (renderer.py:157-167,288-300)."""
    d1, c1, s1 = _cuda_f32(depths1, "depths1"), _cuda_f32(colors1, "colors1"), _cuda_f32(sigma1, "densities1")
    has2 = depths2 is not None
    d2 = _cuda_f32(depths2, "depths2") if has2 else None
    c2 = _cuda_f32(colors2, "colors2") if has2 else None
    s2 = _cuda_f32(sigma2, "densities2") if has2 else None
    g1 = _cuda_f32(segs1, "segs1") if segs1 is not None else None
    g2 = _cuda_f32(segs2, "segs2") if (segs2 is not None and has2) else None
    n, r, n1, _ = d1.shape
    n2 = d2.shape[2] if has2 else 0
    cc = c1.shape[-1]
    cs = g1.shape[-1] if g1 is not None else 0
    dev = d1.device
    S = n1 + n2
    depths = torch.empty((n, r, S, 1), device=dev, dtype=torch.float32)
    colors = torch.empty((n, r, S, cc), device=dev, dtype=torch.float32)
    sigma = torch.empty((n, r, S, 1), device=dev, dtype=torch.float32)
    segs = torch.empty((n, r, S, cs), device=dev, dtype=torch.float32) if cs else None
    with _Guard(d1):
        _lib.check(_lib.load().nfe_unify_samples(_ptr(d1), _ptr(c1), _ptr(g1), _ptr(s1), _ptr(d2), _ptr(c2), _ptr(g2), _ptr(s2), n * r, n1, n2,
                                                 cc, cs, _ptr(depths), _ptr(colors), _ptr(segs), _ptr(sigma), _stream(d1)),
                   "nfe_unify_samples")
    return depths, colors, segs, sigma


# ------------------------------------------------------------------------------- fused forward
PRECISIONS = {"fp32": _lib.PREC_FP32, "bf16x3": _lib.PREC_BF16X3, "bf16": _lib.PREC_BF16}


def precision_of(options):
    """rendering_options['nfe_precision'] -> NFE_PREC_* (decoder MLP arithmetic).  Default: $NFE_DEFAULT_PRECISION, else 'bf16x3'
    — the tensor-core path whose results stay within the path's fp32 tolerance (1e-4) of the reference."""
    default = os.environ.get("NFE_DEFAULT_PRECISION", "bf16x3")
    name = options.get('nfe_precision', default) if options is not None else default
    if name not in PRECISIONS:
        raise RuntimeError(f"nfe_precision must be one of {sorted(PRECISIONS)}, got {name!r}")
    return PRECISIONS[name]


def make_cfg(kind, planes_cl, s_c, s_f, box_warp, white_back=False, density_noise=0.0, stochastic=False, seed=0, offset=0,
             precision=_lib.PREC_FP32, affine=None):
    """affine = (scale [K,96], shift [K,96]) device tensors (K = batch or 1) enables the single-gather identity."""
    _, _, h, w, c = planes_cl.shape
    cfg = NfeRenderCfg(kind, c, h, w, int(s_c), int(s_f), 32, 0 if kind == DEC_OSG else 15, int(bool(white_back)),
                       float(box_warp), float(density_noise), int(bool(stochastic)), seed, offset, precision, None, None, 0)
    if affine is not None:
        scale, shift = affine
        cfg.affine_scale, cfg.affine_shift, cfg.affine_items = scale.data_ptr(), shift.data_ptr(), scale.shape[0]
        cfg._keep = (scale, shift)          # keep the tensors alive as long as the cfg
    return cfg


def workspace_limit_bytes():
    """Upper bound for one nfe_render_fwd workspace ($NFE_WORKSPACE_MB, default 8192).  Larger renders (the
    256^2 x 96+96 x batch-64 sweep would need 158 GB) are split into batch-item / ray-block chunks; the depth
    clamp's global range is combined across the chunks before nfe_finish_depth, so results do not depend on it."""
    import os
    return int(os.environ.get("NFE_WORKSPACE_MB", "8192")) << 20


def render_fwd(cfg, seq_a, seq_b, planes_norm_cl, planes_denorm_cl, origins, dirs, depths_coarse, u_fine,
               finish_depth=True, return_stages=False, keep_workspace=False):
    """Fused forward.  Returns (rgb [N,R,32], seg [N,R,15]|None, depth [N,R,1], wsum [N,R,1], minmax [2][, stages]); rgb is None
    when cfg.geometry_only is set.
    keep_workspace (training): the stages dict also carries views of the per-sample densities / records the
    backward re-reads (sigma_c, rec_c, sigma_f, rec_f) and keeps the workspace alive."""
    o, d = _cuda_f32(origins, "ray_origins"), _cuda_f32(dirs, "ray_directions")
    if o.dim() != 3 or o.shape[-1] != 3 or d.shape != o.shape:
        raise RuntimeError(f"ray_origins / ray_directions: expected matching [N,R,3], got {tuple(o.shape)} and {tuple(d.shape)}")
    n, r, _ = o.shape
    dev = o.device
    dc = _cuda_f32(depths_coarse, "depths_coarse").reshape(n, r, cfg.s_c)
    a = MlpRef(seq_a, dev)
    b = MlpRef(seq_b, dev) if seq_b is not None else None
    image = bool(cfg.image_layout)
    rgb = None if cfg.geometry_only else torch.empty((n, 32, r) if image else (n, r, 32), device=dev, dtype=torch.float32)
    seg = torch.empty((n, cfg.seg_dim, r) if image else (n, r, cfg.seg_dim), device=dev, dtype=torch.float32) if cfg.seg_dim else None
    depth = torch.empty((n, r, 1), device=dev, dtype=torch.float32)
    wsum = torch.empty((n, r, 1), device=dev, dtype=torch.float32)
    minmax = torch.empty(2, device=dev, dtype=torch.float32)
    dfine = torch.empty((n, r, max(cfg.s_f, 1), 1), device=dev, dtype=torch.float32) if return_stages and cfg.s_f else None
    wcoarse = torch.empty((n, r, cfg.s_c - 1, 1), device=dev, dtype=torch.float32) if return_stages and cfg.s_f else None
    lib = _lib.load()
    kept = {}
    any_planes = planes_denorm_cl if planes_denorm_cl is not None else planes_norm_cl     # denorm is absent under the single-gather identity
    shared_planes = any_planes.shape[0] == 1 and n > 1

    def call(i0, i1, r0, r1, mm, finish):
        """rays [r0,r1) of items [i0,i1); a ray sub-range is only used with a single item, so every slice is contiguous"""
        cn, cr = i1 - i0, r1 - r0
        nbytes = lib.nfe_render_workspace_bytes(ctypes.byref(cfg), cn, cr)
        if nbytes < 0:
            raise RuntimeError("nfe_render_workspace_bytes: bad arguments")
        ws = torch.empty(max(int(nbytes), 1), device=dev, dtype=torch.uint8)
        kept["ws"] = ws
        sl = (slice(i0, i1), slice(r0, r1))
        pn = planes_norm_cl if (planes_norm_cl is None or shared_planes) else planes_norm_cl[i0:i1]
        pd = planes_denorm_cl if (planes_denorm_cl is None or shared_planes) else planes_denorm_cl[i0:i1]
        ccfg = cfg
        if (i0, i1, r0, r1) != (0, n, 0, r):
            ccfg = NfeRenderCfg.from_buffer_copy(cfg)
            if cfg.affine_scale and cfg.affine_items == n:             # per-item statistics: shift to this chunk's items
                ccfg.affine_scale, ccfg.affine_shift, ccfg.affine_items = cfg.affine_scale + i0 * 96 * 4, cfg.affine_shift + i0 * 96 * 4, cn
            # the kernels index their Philox streams by the LOCAL sample number: give every workspace chunk its own offsets
            # (all 64 bits of the offset enter the counter; torch's generator advances it by 16 per call, far below 2^40),
            # or all chunks would draw the same jitter and density noise
            ccfg.offset = cfg.offset + (len(kept.setdefault("chunks", [])) << 40)
            kept["chunks"].append((i0, i1, r0, r1))
        oo, dd, dcc = o[sl].contiguous(), d[sl].contiguous(), dc[sl].contiguous()     # no copies: whole items, or rays of one item
        outs = [rgb, seg, depth, wsum]
        if image and cr != r:
            raise RuntimeError("render_fwd: image-layout outputs cannot be split into ray blocks; raise NFE_WORKSPACE_MB")
        map_sl = (slice(i0, i1),) if image else sl            # image layout [n, C, r]: only whole items can be sliced
        views = [None if rgb is None else rgb[map_sl], None if seg is None else seg[map_sl], depth[sl], wsum[sl]]
        direct = all(v is None or v.is_contiguous() for v in views)
        bufs = views if direct else [None if v is None else torch.empty_like(v) for v in views]
        rc = lib.nfe_render_fwd(ctypes.byref(ccfg), a.ref(), b.ref() if b else None, _ptr(pn), _ptr(pd), (pn if pd is None else pd).shape[0], _ptr(oo), _ptr(dd), cn, cr,
                                _ptr(dcc), _ptr(u_fine), _ptr(bufs[0]), _ptr(bufs[1]), _ptr(bufs[2]), _ptr(bufs[3]), _ptr(mm), int(bool(finish)),
                                _ptr(dfine), _ptr(wcoarse), _ptr(ws), int(nbytes), _stream(o))
        _lib.check(rc, "nfe_render_fwd")
        if not direct:
            for v, bf in zip(views, bufs):
                if v is not None:
                    v.copy_(bf)

    with _Guard(o):
        limit = workspace_limit_bytes()
        plan_cfg = cfg
        if cfg.geometry_only and (cfg.stochastic or cfg.density_noise > 0):
            # every chunk draws its jitter and density noise from its own Philox offset: a geometry-only render whose draws
            # must match the full render's splits where the full render would, and allocates only its smaller workspace
            plan_cfg = NfeRenderCfg.from_buffer_copy(cfg)
            plan_cfg.geometry_only = 0
        per_item = lib.nfe_render_workspace_bytes(ctypes.byref(plan_cfg), 1, r) if n and r else 0
        if n * per_item <= limit or n * r == 0 or keep_workspace:
            call(0, n, 0, r, minmax, finish_depth)
        else:
            if return_stages:
                raise RuntimeError("render_fwd: stage taps are not available for renders split into workspace chunks")
            parts = []
            if per_item <= limit:                                   # groups of whole items
                step = max(1, limit // per_item)
                chunks = [(i, min(i + step, n), 0, r) for i in range(0, n, step)]
            else:                                                   # ray blocks inside each item
                per_ray = max(1, per_item // r)
                rstep = max(1, limit // per_ray)
                chunks = [(i, i + 1, q, min(q + rstep, r)) for i in range(n) for q in range(0, r, rstep)]
            for (i0, i1, r0, r1) in chunks:
                mm = torch.empty(2, device=dev, dtype=torch.float32)
                call(i0, i1, r0, r1, mm, False)
                parts.append(mm)
            mms = torch.stack(parts)
            minmax = torch.stack([mms[:, 0].min(), mms[:, 1].max()])
            if finish_depth:
                _lib.check(lib.nfe_finish_depth(_ptr(depth), depth.numel(), _ptr(minmax), _stream(o)), "nfe_finish_depth")
    if return_stages:
        stages = {"depths_fine": dfine, "weights_coarse": wcoarse}
        if keep_workspace and n * r:
            offs = (ctypes.c_int64 * 4)()
            _lib.check(lib.nfe_render_workspace_layout(ctypes.byref(cfg), n, r, offs), "nfe_render_workspace_layout")
            ws = kept["ws"]

            def view(off, *shape):
                count = 1
                for s_ in shape:
                    count *= s_
                return ws[off:off + 4 * count].view(torch.float32).view(*shape)
            stages.update(workspace=ws, sigma_c=view(offs[0], n * r, cfg.s_c), rec_c=view(offs[1], n * r, cfg.s_c, 48))
            if cfg.s_f:
                stages.update(sigma_f=view(offs[2], n * r, cfg.s_f), rec_f=view(offs[3], n * r, cfg.s_f, 48))
        return rgb, seg, depth, wsum, minmax, stages
    return rgb, seg, depth, wsum, minmax


def finish_depth(depth, minmax):
    with _Guard(depth):
        _lib.check(_lib.load().nfe_finish_depth(_ptr(depth), depth.numel(), _ptr(minmax), _stream(depth)), "nfe_finish_depth")
    return depth


def run_model_fwd(cfg, seq_a, seq_b, planes_norm_cl, planes_denorm_cl, coords, sigma_only=False):
    co = _cuda_f32(coords, "sample_coordinates")
    if co.dim() != 3 or co.shape[-1] != 3:
        raise RuntimeError(f"sample_coordinates: expected [N,M,3], got {tuple(co.shape)}")
    n, m, _ = co.shape
    dev = co.device
    a = MlpRef(seq_a, dev)
    b = MlpRef(seq_b, dev) if seq_b is not None else None
    cfg.sigma_only = int(bool(sigma_only))
    rgb = torch.empty((n, m, 32), device=dev, dtype=torch.float32) if not sigma_only else None
    sigma = torch.empty((n, m, 1), device=dev, dtype=torch.float32)
    seg = torch.empty((n, m, 15), device=dev, dtype=torch.float32) if (cfg.seg_dim and not sigma_only) else None
    any_planes = planes_denorm_cl if planes_denorm_cl is not None else planes_norm_cl
    with _Guard(co):
        rc = _lib.load().nfe_run_model_fwd(ctypes.byref(cfg), a.ref(), b.ref() if b else None, _ptr(planes_norm_cl), _ptr(planes_denorm_cl),
                                           any_planes.shape[0], _ptr(co), n, m, _ptr(rgb), _ptr(sigma), _ptr(seg), None, 0, _stream(co))
    _lib.check(rc, "nfe_run_model_fwd")
    if sigma_only:
        return {"sigma": sigma}
    out = {"rgb": rgb, "sigma": sigma}
    if seg is not None:
        out["seg"] = seg
    return out
