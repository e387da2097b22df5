"""Geometry-only renders (rendering_options['nfe_geometry_only']): the semantic masks, depth and weight sums of a view without the
appearance branch.  seg, depth and wsum must be bit-identical (torch.equal) to those of the full render of the same inputs — the
compositing weights, the importance resampling and the seg sums depend on the densities and the geo_net / seg_net logits alone,
and the geometry-only kernels compute those with the same arithmetic in the same order — and rgb is None."""
import numpy as np
import pytest
import torch

import synth_inputs as synth
from _util import golden
from test_gpu_full_size import _check_maps, _planes
from test_gpu_parity import N, T, PlainDecoder, torch_decoder

pytestmark = pytest.mark.gpu
TAGS = {"dis": "dis_12_12", "seg": "seg_12_12", "osg": "osg_12_12"}


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def _setup(dev, kind, flow, n=2, hw=32, res=16, seed=21):
    """(renderer, plane args, decoder, origins, dirs).  flow 'package': normalize_plane of this package (the full render takes the
    single-gather identity in the tensor-core modes); 'foreign': plain torch normalisation (no provenance: the full render gathers
    both plane sets); 'staged': a decoder the fused path does not recognise."""
    from nerffaceediting_b200 import triplane
    from nerffaceediting_b200.ray_sampler import RaySampler
    from nerffaceediting_b200.renderer import DisentangledImportanceRenderer, ImportanceRenderer
    g = golden("render_small")
    dec = torch_decoder(g, f"{TAGS[kind]}.dec", kind, 1.0, dev)
    if flow == "staged":
        dec = PlainDecoder(dec)
    raw = T(synth.hash_normal(seed, (n, 96, hw, hw)) * np.float32(1.5) - np.float32(0.3), dev)
    c2w, k = synth.camera_sweep(n)
    o, d = RaySampler()(c2w.to(dev), k.to(dev), res)
    v = lambda t: t.view(n, 3, 32, hw, hw)
    if kind == "osg":
        return ImportanceRenderer(), (v(raw),), dec, o, d
    if flow == "foreign":
        mean, std = raw.mean(dim=(-1, -2), keepdim=True), raw.var(dim=(-1, -2), keepdim=True).sqrt()
        norm = (raw - mean) / (std + 1e-8)
    else:
        norm = triplane.normalize_plane(raw)[0]
    return DisentangledImportanceRenderer(), (v(norm), v(raw)), dec, o, d


def _assert_geometry(full, geo, kind):
    """geo = (None, seg, depth, wsum) / (None, depth, wsum) with the full render's maps, bit for bit."""
    assert len(geo) == len(full) and geo[0] is None and full[0] is not None
    for a, b in zip(full[1:], geo[1:]):
        assert b.shape == a.shape and b.dtype == a.dtype and torch.equal(a, b)
    if kind != "osg":
        assert geo[1].shape[-1] == 15 or geo[1].shape[1] == 15


@pytest.mark.parametrize("flow", ["package", "foreign", "staged"])
@pytest.mark.parametrize("precision", ["fp32", "bf16x3", "bf16"])
@pytest.mark.parametrize("kind", ["dis", "seg", "osg"])
def test_geometry_only_equals_full_render(dev, kind, precision, flow):
    """Every decoder x precision x plane flow, in deterministic mode, stochastic mode with density noise (same seed), with a
    white background and with a single pass (depth_resolution_importance = 0)."""
    from nerffaceediting_b200 import ops
    if kind == "osg" and flow == "foreign":
        pytest.skip("the OSG decoder reads one plane set: no normalisation flow")
    ren, args, dec, o, d = _setup(dev, kind, flow)
    base = dict(synth.FFHQ_RENDERING_OPTIONS, depth_resolution=24, depth_resolution_importance=24, nfe_precision=precision)
    cases = {
        "deterministic": dict(base, nfe_deterministic=True),
        "stochastic_noise": dict(base, density_noise=0.5),
        "white_back": dict(base, nfe_deterministic=True, white_back=True),
        "single_pass": dict(base, nfe_deterministic=True, depth_resolution=40, depth_resolution_importance=0),
    }
    with torch.no_grad():
        for name, opts in cases.items():
            torch.cuda.manual_seed(7)
            full = ren(*args, dec, o, d, opts)
            ops.path_counts(reset=True)
            torch.cuda.manual_seed(7)
            geo = ren(*args, dec, o, d, dict(opts, nfe_geometry_only=True))
            paths = ops.path_counts(reset=True)
            _assert_geometry(full, geo, kind)
            if flow == "staged":
                assert paths.get("render:staged", 0) == 1, (name, paths)
            else:
                assert paths.get("render:geometry-only", 0) == 1, (name, paths)
                if kind == "dis":
                    # only the normalised planes are staged (a hit when normalize_plane staged them, a miss otherwise)
                    assert sum(v for k, v in paths.items() if k.startswith("staging:")) == 1, (name, paths)
    assert not torch.equal(full[-1], torch.zeros_like(full[-1]))


@pytest.mark.parametrize("precision", ["fp32", "bf16x3"])
def test_geometry_only_image_layout(dev, precision):
    """nfe_image_layout: seg_image / depth_image of a geometry-only render are the full render's, rgb stays None."""
    opts = dict(synth.FFHQ_RENDERING_OPTIONS, depth_resolution=24, depth_resolution_importance=24, nfe_deterministic=True,
                nfe_precision=precision, nfe_image_layout=True)
    n, res = 2, 16
    with torch.no_grad():
        for kind in ("dis", "osg"):
            ren, args, dec, o, d = _setup(dev, kind, "package", n=n, res=res)
            full = ren(*args, dec, o, d, opts)
            geo = ren(*args, dec, o, d, dict(opts, nfe_geometry_only=True))
            _assert_geometry(full, geo, kind)
            flat = ren(*args, dec, o, d, dict(opts, nfe_image_layout=False, nfe_geometry_only=True))
            if kind == "dis":
                assert geo[1].shape == (n, 15, res, res) and geo[2].shape == (n, 1, res, res)
                assert torch.equal(geo[1], flat[1].permute(0, 2, 1).reshape(n, 15, res, res))
            assert torch.equal(geo[-2], flat[-2].reshape(n, 1, res, res)) and torch.equal(geo[-1], flat[-1])


@pytest.mark.parametrize("precision", ["fp32", "bf16x3"])
def test_geometry_only_workspace_chunks(dev, monkeypatch, precision):
    """A geometry-only render split into workspace chunks (groups of items, ray blocks of one item) equals the unsplit one."""
    ren, args, dec, o, d = _setup(dev, "dis", "package", n=3, res=32)
    opts = dict(synth.FFHQ_RENDERING_OPTIONS, depth_resolution=24, depth_resolution_importance=24, nfe_deterministic=True,
                nfe_precision=precision, nfe_geometry_only=True)
    with torch.no_grad():
        whole = ren(*args, dec, o, d, opts)
        monkeypatch.setenv("NFE_WORKSPACE_MB", "8")        # one item needs ~3.5 MB: groups of two items
        by_items = ren(*args, dec, o, d, opts)
        monkeypatch.setenv("NFE_WORKSPACE_MB", "2")        # less than one item: ray blocks
        by_rays = ren(*args, dec, o, d, opts)
    for a, b, c in zip(whole[1:], by_items[1:], by_rays[1:]):
        assert torch.equal(a, b) and torch.equal(a, c)


@pytest.mark.parametrize("precision", ["fp32", "bf16x3"])
def test_geometry_only_stochastic_workspace_chunks(dev, monkeypatch, precision):
    """Stochastic sampling with density noise, at a workspace bound where the full render splits into chunks (and so gives each
    chunk its own Philox offset) but the smaller geometry-only workspace alone would not: the geometry-only render splits the same
    way and stays bit-identical to the full render."""
    ren, args, dec, o, d = _setup(dev, "dis", "package", n=3, res=32)
    opts = dict(synth.FFHQ_RENDERING_OPTIONS, depth_resolution=24, depth_resolution_importance=24, density_noise=0.5,
                nfe_precision=precision)
    with torch.no_grad():
        torch.cuda.manual_seed(5)
        unsplit = ren(*args, dec, o, d, opts)
        monkeypatch.setenv("NFE_WORKSPACE_MB", "20")       # full: ~9.8 MB per item -> chunks of two items; geometry: ~3.5 MB
        torch.cuda.manual_seed(5)
        full = ren(*args, dec, o, d, opts)
        torch.cuda.manual_seed(5)
        geo = ren(*args, dec, o, d, dict(opts, nfe_geometry_only=True))
    assert not torch.equal(full[-1], unsplit[-1])          # the split changed the draws: the case under test is exercised
    _assert_geometry(full, geo, "dis")


@pytest.mark.parametrize("precision", ["fp32", "bf16x3"])
def test_geometry_only_shared_planes_many_poses(dev, precision):
    """One plane set broadcast over several poses (the video-sweep pattern): equals the expanded batch and the full render."""
    from nerffaceediting_b200 import triplane
    from nerffaceediting_b200.ray_sampler import RaySampler
    from nerffaceediting_b200.renderer import DisentangledImportanceRenderer
    g = golden("render_small")
    dec = torch_decoder(g, "dis_12_12.dec", "dis", 1.0, dev)
    raw = T(synth.hash_normal(9, (1, 96, 32, 32)), dev)
    norm = triplane.normalize_plane(raw)[0].view(1, 3, 32, 32, 32)
    planes = raw.view(1, 3, 32, 32, 32)
    c2w, k = synth.camera_sweep(5)
    o, d = RaySampler()(c2w.to(dev), k.to(dev), 16)
    opts = dict(synth.FFHQ_RENDERING_OPTIONS, depth_resolution=24, depth_resolution_importance=24, nfe_deterministic=True,
                nfe_precision=precision)
    ren = DisentangledImportanceRenderer()
    with torch.no_grad():
        full = ren(norm, planes, dec, o, d, opts)
        geo = ren(norm, planes, dec, o, d, dict(opts, nfe_geometry_only=True))
        expanded = ren(norm.expand(5, -1, -1, -1, -1), planes.expand(5, -1, -1, -1, -1), dec, o, d, dict(opts, nfe_geometry_only=True))
    _assert_geometry(full, geo, "dis")
    for a, b in zip(geo[1:], expanded[1:]):
        assert torch.equal(a, b)


def test_geometry_only_cuda_graph_replay(dev):
    """graphs.capture of RaySampler -> normalize_plane -> geometry-only render: replays are bit-identical to the eager call."""
    from nerffaceediting_b200 import graphs, triplane
    from nerffaceediting_b200.ray_sampler import RaySampler
    from nerffaceediting_b200.renderer import DisentangledImportanceRenderer
    g = golden("render_small")
    dec = torch_decoder(g, "dis_12_12.dec", "dis", 1.0, dev)
    raw = T(synth.hash_normal(21, (2, 96, 32, 32)), dev)
    c2w, k = synth.camera_sweep(2)
    c2w, k = c2w.to(dev), k.to(dev)
    opts = dict(synth.FFHQ_RENDERING_OPTIONS, depth_resolution=12, depth_resolution_importance=12, nfe_deterministic=True,
                nfe_geometry_only=True)
    sampler, ren = RaySampler(), DisentangledImportanceRenderer()

    def step():
        o, d = sampler(c2w, k, 16)
        norm, _, _ = triplane.normalize_plane(raw)
        return ren(norm.view(2, 3, 32, 32, 32), raw.view(2, 3, 32, 32, 32), dec, o, d, opts)

    call = graphs.capture(step)
    assert call.kernels >= 6 and call.outputs[0] is None
    with torch.no_grad():
        for seed in (21, 22):
            raw.copy_(T(synth.hash_normal(seed, (2, 96, 32, 32)), dev))
            replayed = [t.clone() for t in call()[1:]]
            eager = step()
            assert eager[0] is None
            for a, b in zip(replayed, eager[1:]):
                assert torch.equal(a, b), seed


def test_geometry_only_refuses_autograd(dev):
    """Geometry-only renders have no backward: a differentiable call raises, naming the option."""
    ren, args, dec, o, d = _setup(dev, "dis", "package")
    opts = dict(synth.FFHQ_RENDERING_OPTIONS, depth_resolution=12, depth_resolution_importance=12, nfe_deterministic=True,
                nfe_geometry_only=True)
    frozen = _setup(dev, "dis", "package")[2].requires_grad_(False)
    ren(*args, frozen, o, d, opts)               # nothing requires grad: renders
    with pytest.raises(RuntimeError, match="nfe_geometry_only"):
        ren(args[0], args[1].clone().requires_grad_(), frozen, o, d, opts)      # the planes alone require grad
    with pytest.raises(RuntimeError, match="nfe_geometry_only"):
        ren(*args, dec, o, d, opts)              # the decoder's parameters alone require grad
    ren_s, args_s, dec_s, o, d = _setup(dev, "dis", "staged")
    with pytest.raises(RuntimeError, match="nfe_geometry_only"):
        ren_s(*args_s, dec_s, o, d, opts)


def test_geometry_only_config3_vs_reference(dev):
    """BASELINE configs[2] (batch 32, 256^2 planes, 128^2 rays, statistics rolled by one item, 48+48) against the reference's own
    render_c3 fixture: seg and depth within the full-size tolerances.  Normalised in plain torch ops (the unpatched-generator flow:
    no provenance); the geometry-only render reads the normalised planes alone either way."""
    from nerffaceediting_b200 import ops
    from nerffaceediting_b200.ray_sampler import RaySampler
    from nerffaceediting_b200.renderer import DisentangledImportanceRenderer
    g = golden("render_c3")
    n, hw, res, stride = 32, 256, int(g["res"]), int(g["ray_stride"])
    raw = _planes(int(g["planes_seed"]), n, dev)
    dec = torch_decoder(g, "dec", "dis", 1.0, dev)
    opts = dict(synth.FFHQ_RENDERING_OPTIONS, nfe_deterministic=True, nfe_geometry_only=True)
    ops.path_counts(reset=True)
    with torch.no_grad():
        o, d = RaySampler()(T(g["cam2world"], dev), T(g["intrinsics"], dev), res)
        mean, std = raw.mean(dim=(-1, -2), keepdim=True), raw.var(dim=(-1, -2), keepdim=True).sqrt()
        norm = (raw - mean) / (std + 1e-8)
        planes = norm * std.roll(1, 0) + mean.roll(1, 0)
        del raw
        rgb, seg, depth, wsum = DisentangledImportanceRenderer()(norm.view(n, 3, 32, hw, hw), planes.view(n, 3, 32, hw, hw), dec, o, d, opts)
    assert rgb is None and seg.shape == (n, res * res, 15)
    paths = ops.path_counts()
    assert paths.get("render:geometry-only", 0) == 1 and paths.get("staging:miss", 0) == 1, paths
    for name, t in (("seg", seg), ("depth", depth), ("wsum", wsum)):
        _check_maps(N(t[:, ::stride]), g[name], f"geometry.{name}")
