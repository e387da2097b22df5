"""The render and run_model backward kernels (march_bwd_kernel, field_bwd_kernel<KIND, AFFINE>, nfe_planes_from_channel_last)
against float64 autograd through tests/_torch_render.py, the plain-torch restatement of the reference that
test_torch_render_reference.py pins to the reference's own gradients.  The cases sit where the three golden shapes do not
reach: per-pass sample counts that are not multiples of 128 with item boundaries inside tiles, one plane set broadcast over
the batch, samples on and beyond the box faces, rays that miss the box, white background, disparity sampling, a single pass,
192 and 768 merged samples, opaque and empty rays, run_model points on texel centres and box faces, and the single-gather
backward through its statistics.

Each render runs under autograd with nfe_deterministic=True.  The coarse and fine depths its fused forward used are captured
from ops.render_fwd and handed to the restatement, which runs in float64 on the GPU from the same planes and parameters.  The
loss is a sum of seeded random projections of every output.  Bars are test_gpu_backward.py's: rel_err < 1e-4 (fp32) and
< 2e-4 (bf16x3) for every gradient, elem_err(floor=1e-2) < 1e-3 for plane gradients, rel_err < 1e-4 for the forward outputs.
The measured errors are attached to each test's report as user properties (pytest --junitxml with junit_family=legacy).
Two cases, limited by float32 arithmetic, also measure the restatement in float32; see FLOAT32_LIMITED."""
import math

import numpy as np
import pytest
import torch

import _torch_render as tr
import synth_inputs as synth
from _util import elem_err, golden, rel_err
from test_gpu_parity import torch_decoder

pytestmark = pytest.mark.gpu
TOL = {"fp32": 1e-4, "bf16x3": 2e-4}
PLANE_ELEM_TOL = 1e-3
# Cases where float32 arithmetic itself, not the kernel, limits the agreement with float64 also run the restatement in
# float32 from the same inputs (the reference's formulation at the kernel's precision).  There each bar becomes
# max(bar, 2 x the float32 restatement's own error against float64): the kernel must be as close to float64 as the reference
# evaluated in float32 is, within a factor of two.  Measured on a B200 before this rule (kernel / float32 restatement):
#   osg-fp32, density-output bias, a signed sum over 26 k samples per pass: rel_err 1.12e-4 and 1.15e-4 (two runs; the
#     library-GEMM backward 1.17e-4) / 9.6e-5;
#   samples-768, plane gradient element-wise, 767 intervals of float32 transmittance: elem_err 1.11e-3 / 1.35e-3.
FLOAT32_LIMITED = {"osg-fp32", "samples-768"}
DEC_SOURCES = {"dis": ("backward", "dis.dec"), "osg": ("backward", "osg.dec"), "seg": ("run_model_bwd", "seg_all.dec")}


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@pytest.fixture
def captured(monkeypatch):
    """The depths each fused render forward used: [(depths_coarse [N,R,S_c,1], depths_fine [N,R,S_f,1] or None)]."""
    from nerffaceediting_b200 import ops
    seen = []
    real = ops.render_fwd

    def spy(cfg, seq_a, seq_b, planes_norm_cl, planes_denorm_cl, origins, dirs, depths_coarse, u_fine, **taps):
        out = real(cfg, seq_a, seq_b, planes_norm_cl, planes_denorm_cl, origins, dirs, depths_coarse, u_fine, **taps)
        fine = out[5]["depths_fine"] if taps.get("return_stages") else None
        seen.append((depths_coarse.detach().clone(), None if fine is None else fine.detach().clone()))
        return out
    monkeypatch.setattr(ops, "render_fwd", spy)
    return seen


def _decoder(kind, dev):
    name, prefix = DEC_SOURCES[kind]
    return torch_decoder(golden(name), prefix, kind, 1.0, dev)


def _planes(seed, n, h, w, dev):
    """(norm, raw) [n,3,32,h,w]: raw planes and their normalisation by the reference's formula in plain torch."""
    raw = torch.from_numpy(synth.hash_normal(seed, (n, 96, h, w)) * np.float32(1.5) - np.float32(0.3)).to(dev)
    mean, std = raw.mean(dim=(-1, -2), keepdim=True), raw.var(dim=(-1, -2), keepdim=True).sqrt()
    return ((raw - mean) / (std + 1e-8)).view(n, 3, 32, h, w), raw.view(n, 3, 32, h, w)


def _rays(n, res, dev, radius=2.7, fov=18.837):
    from nerffaceediting_b200.ray_sampler import RaySampler
    yaw = [0.4 * (2 * i / max(n - 1, 1) - 1) for i in range(n)]
    pitch = [0.25 * (2 * i / max(n - 1, 1) - 1) for i in range(n)]
    c2w = synth.look_at_cam2world([math.pi / 2 + y for y in yaw], [math.pi / 2 + p for p in pitch], radius=radius)
    k = synth.fov_to_intrinsics(fov).unsqueeze(0).repeat(n, 1, 1)
    with torch.no_grad():
        return RaySampler()(c2w.to(dev), k.to(dev), res)


def _projections(shapes, seed, dev):
    gen = torch.Generator().manual_seed(seed)
    return [torch.randn(s, generator=gen, dtype=torch.float64).to(dev) for s in shapes]


class Report:
    """Asserts one comparison and records its measured error as a user property of the test.  `f32`: the same quantity from
    the restatement in float32 (FLOAT32_LIMITED cases), which widens the bar to twice its own error."""

    def __init__(self, record_property):
        self.record = record_property

    def _check(self, metric, fn, what, got, want, tol, f32):
        want = want.detach().cpu().numpy()
        e = fn(got.detach().cpu().numpy(), want)
        self.record(f"{metric} {what}", f"{e:.3g}")
        if f32 is not None:
            e32 = fn(f32.detach().cpu().numpy(), want)
            self.record(f"{metric} {what} (float32 restatement)", f"{e32:.3g}")
            tol = max(tol, 2 * e32)
        assert e < tol, (what, e, tol)

    def rel(self, what, got, want, tol, f32=None):
        self._check("rel_err", rel_err, what, got, want, tol, f32)

    def elem(self, what, got, want, tol, f32=None):
        self._check("elem_err", lambda a, b: elem_err(a, b, floor=1e-2), what, got, want, tol, f32)


def _compare_grads(rep, tag, precision, leaves, dec, ref_dec, f32=None):
    """leaves: [(name, kernel-side leaf, restatement leaf, is_plane)]; f32: {name: float32 restatement gradient} or None."""
    tol = TOL[precision]
    f32 = f32 or {}
    for name, a, b, plane in leaves:
        assert a.grad is not None and b.grad is not None and a.grad.shape == b.grad.shape, name
        rep.rel(f"{tag} {name}", a.grad, b.grad, tol, f32.get(name))
        if plane:
            rep.elem(f"{tag} {name}", a.grad, b.grad, PLANE_ELEM_TOL, f32.get(name))
    for name, p in dec.named_parameters():
        rep.rel(f"{tag} dec.{name}", p.grad, ref_dec.params[name].grad, tol, f32.get(f"dec.{name}"))


def _render_case(dev, captured, rep, tag, kind, precision, norm, planes, o, d, opts, dec=None, zero_depth_rays=None):
    """Render with the package under autograd and with the restatement in float64 from the captured depths; compare the
    forward outputs and the gradients of the plane tensors and every decoder parameter.  zero_depth_rays(depths_coarse,
    depths_fine) -> [N,R,1] bool: rays whose depth is left out of the loss and of the depth comparison."""
    from nerffaceediting_b200.renderer import DisentangledImportanceRenderer, ImportanceRenderer
    dec = dec if dec is not None else _decoder(kind, dev)
    opts = dict(synth.FFHQ_RENDERING_OPTIONS, **opts, nfe_deterministic=True, nfe_precision=precision)
    n, r, _ = o.shape
    leaves = []
    p_k = planes.detach().clone().requires_grad_(True)
    p_r = planes.detach().double().requires_grad_(True)
    leaves.append(("g_planes", p_k, p_r, True))
    n_k = n_r = None
    if kind != "osg":
        n_k = norm.detach().clone().requires_grad_(True)
        n_r = norm.detach().double().requires_grad_(True)
        if kind == "dis":
            leaves.append(("g_norm", n_k, n_r, True))
    captured.clear()
    if kind == "osg":
        rgb, depth, wsum = ImportanceRenderer()(p_k, dec, o, d, opts)
        seg = None
    else:
        rgb, seg, depth, wsum = DisentangledImportanceRenderer()(n_k, p_k, dec, o, d, opts)
    assert len(captured) == 1
    dc, df = captured[0]
    if callable(zero_depth_rays):
        zero_depth_rays = zero_depth_rays(dc, df)
    ref_dec = tr.Decoder(dec, torch.float64, dev)
    want = tr.render(ref_dec, n_r, p_r, o, d, dc, df, opts['box_warp'], opts['white_back'])
    proj = _projections([(n, r, 32), (n, r, 15), (n, r, 1), (n, r, 1)], 4242, dev)
    if zero_depth_rays is not None:
        proj[2] = torch.where(zero_depth_rays, torch.zeros_like(proj[2]), proj[2])
    names = ("rgb", "seg", "depth", "wsum")
    got = (rgb, seg, depth, wsum)
    for nm, a, b in zip(names, got, want):
        if a is None:
            continue
        if nm == "depth" and zero_depth_rays is not None:
            keep = ~zero_depth_rays
            rep.rel(f"{tag} out.depth", a[keep], b[keep], 1e-4)
        else:
            rep.rel(f"{tag} out.{nm}", a, b, 1e-4)
    sum((a.double() * w).sum() for a, w in zip(got, proj) if a is not None).backward(retain_graph=zero_depth_rays is not None)
    sum((a * w).sum() for a, w in zip(want, proj) if a is not None).backward()
    f32 = None
    if tag in FLOAT32_LIMITED:
        dec32 = tr.Decoder(dec, torch.float32, dev)
        p32 = planes.detach().clone().requires_grad_(True)
        n32 = None if norm is None else norm.detach().clone().requires_grad_(True)
        want32 = tr.render(dec32, n32, p32, o, d, dc, df, opts['box_warp'], opts['white_back'])
        sum((a.double() * w).sum() for a, w in zip(want32, proj) if a is not None).backward()
        f32 = {"g_planes": p32.grad, "g_norm": None if n32 is None else n32.grad, **{f"dec.{k}": v.grad for k, v in dec32.params.items()}}
    _compare_grads(rep, tag, precision, leaves, dec, ref_dec, f32)
    return dict(out=got, want=want, dc=dc, df=df, planes=p_k, norm=n_k, dec=dec, empty=zero_depth_rays)


GRID = dict(n=3, h=40, w=24, res=19, s=24)       # 361 rays x 24 samples = 8664 per item and pass: not a multiple of 128
RENDER_CASES = {f"{kind}-{prec}": (kind, prec) for kind in ("osg", "dis", "seg") for prec in ("fp32", "bf16x3")}


@pytest.mark.parametrize("case", list(RENDER_CASES))
def test_render_backward_multi_tile(dev, captured, record_property, case):
    """Every decoder kind on the multi-tile path: ragged last tile, item boundaries inside tiles, non-square planes."""
    kind, precision = RENDER_CASES[case]
    norm, planes = _planes(401, GRID["n"], GRID["h"], GRID["w"], dev)
    o, d = _rays(GRID["n"], GRID["res"], dev)
    _render_case(dev, captured, Report(record_property), case, kind, precision, norm, planes, o, d,
                 dict(depth_resolution=GRID["s"], depth_resolution_importance=GRID["s"]))


@pytest.mark.parametrize("kind", ["osg", "dis"])
def test_render_backward_broadcast_planes(dev, captured, record_property, kind):
    """One plane set [1,3,32,H,W] under 3 ray items: every item scatters into the same plane gradient."""
    norm, planes = _planes(402, 1, 32, 28, dev)
    o, d = _rays(3, 17, dev)
    _render_case(dev, captured, Report(record_property), f"broadcast-{kind}", kind, "fp32", norm, planes, o, d,
                 dict(depth_resolution=24, depth_resolution_importance=24))


def test_render_backward_box_edges(dev, captured, record_property):
    """box_warp = 1.6 with the camera pulled in to 1.6 from the centre, so that the samples enter and leave the box through its
    faces; then 'auto' limits with a wide camera whose corner rays miss the box (the _auto_limits patch)."""
    from nerffaceediting_b200 import math_utils
    rep = Report(record_property)
    norm, planes = _planes(403, 2, 24, 24, dev)
    o, d = _rays(2, 16, dev, radius=1.6)
    res = _render_case(dev, captured, rep, "box-edges fixed", "dis", "fp32", norm, planes, o, d,
                       dict(depth_resolution=24, depth_resolution_importance=24, box_warp=1.6, ray_start=0.1, ray_end=2.8))
    pts = o.unsqueeze(-2) + res["dc"] * d.unsqueeze(-2)
    inside = (pts.abs() <= 0.8).all(-1)
    assert inside.any() and (~inside).any(), "the coarse samples must lie on both sides of the box faces"
    o, d = _rays(2, 16, dev, fov=60.0)
    t0, t1 = math_utils.get_ray_limits_box(o, d, box_side_length=1.6)
    assert (t1 <= t0).any() and (t1 > t0).any(), "some rays must miss the box and some hit it"
    _render_case(dev, captured, rep, "box-edges auto", "dis", "fp32", norm, planes, o, d,
                 dict(depth_resolution=24, depth_resolution_importance=24, box_warp=1.6, ray_start='auto', ray_end='auto'))


OPTION_CASES = {
    "white-back": dict(depth_resolution=24, depth_resolution_importance=24, white_back=True),
    "disparity": dict(depth_resolution=24, depth_resolution_importance=16, disparity_space_sampling=True),
    "single-pass": dict(depth_resolution=40, depth_resolution_importance=0),
}


@pytest.mark.parametrize("case", list(OPTION_CASES))
def test_render_backward_options(dev, captured, record_property, case):
    """White background and disparity sampling beyond the goldens' 8^2 rays; a single pass (s2 == 0 in both backward kernels)."""
    norm, planes = _planes(404, GRID["n"], GRID["h"], GRID["w"], dev)
    o, d = _rays(GRID["n"], GRID["res"], dev)
    _render_case(dev, captured, Report(record_property), case, "dis", "fp32", norm, planes, o, d, OPTION_CASES[case])


@pytest.mark.parametrize("case,samples,res", [("samples-192", 96, 5), ("samples-768", 384, 3)])
def test_render_backward_many_samples(dev, captured, record_property, case, samples, res):
    """192 merged samples (several intervals per lane chunk) and 768 (the maximum; the backward's warp-count fallback)."""
    norm, planes = _planes(405, 2, 32, 32, dev)
    o, d = _rays(2, res, dev)
    _render_case(dev, captured, Report(record_property), case, "dis", "fp32", norm, planes, o, d,
                 dict(depth_resolution=samples, depth_resolution_importance=samples))


def _sigma_direction(dec, sign):
    """A unit channel vector e_k (times +-1) along which the density output of the geometry net grows fastest (sign=+1) or
    falls fastest (sign=-1) once the features are large: the asymptotic slope of FC . Softplus . FC."""
    a, b = dec.geo_net[0], dec.geo_net[2]
    w1 = (a.weight * a.weight_gain).detach().double()
    w2 = (b.weight[0] * b.weight_gain).detach().double()
    cand = torch.cat([torch.eye(32, dtype=torch.float64), -torch.eye(32, dtype=torch.float64)]).to(w1.device)
    slope = (torch.relu(cand @ w1.t()) * w2).sum(1) * sign
    return cand[int(slope.argmax())].float(), float(slope.max())


def test_render_backward_opaque_and_empty(dev, captured, record_property):
    """Three items of one render: item 0 as drawn, item 1 opaque (density above 1000 at every sample: alpha == 1 in float32,
    where the backward divides by 1 - alpha + 1e-10), item 2 empty (density below -30 at every sample: float32 weight totals
    of 0, a depth that is the global maximum and carries no gradient).  The decoder is shared by the items, so the densities
    are pushed per item through the normalised planes: a constant offset along the channel the geometry net's density is
    most sensitive to.  The rays stay inside the box, so every sample sees the whole offset.

    Rays whose float32 weight total is 0 keep a finite float64 depth; that difference is a dtype effect, so their depth is
    left out of the loss and of the depth comparison, and checked on its own."""
    rep = Report(record_property)
    n, hw = 3, 24
    norm, planes = _planes(406, n, hw, hw, dev)
    o, d = _rays(n, 12, dev, fov=12.0)
    opts = dict(depth_resolution=24, depth_resolution_importance=24, ray_start=2.45, ray_end=2.95)
    depths = torch.linspace(opts['ray_start'], opts['ray_end'], 97, device=dev)
    pts = o.unsqueeze(-2) + depths.view(1, 1, -1, 1) * d.unsqueeze(-2)
    assert float(pts.abs().max()) < 0.5 - 1.0 / hw, "every sample must lie inside the box, away from its faces"
    dec = _decoder("dis", dev)
    ref32 = tr.Decoder(dec, torch.float32, dev)
    norm = norm.clone()
    for item, sign, ok in ((1, 1, lambda s: float(s.min()) > 1000), (2, -1, lambda s: float(s.max()) < -30)):
        u, slope = _sigma_direction(dec, sign)
        assert slope > 0
        c = 1.0
        while True:
            trial = norm[item:item + 1] + c * u.view(1, 1, 32, 1, 1)
            with torch.no_grad():
                sig = tr.run_model(ref32, trial, planes[item:item + 1], pts[item:item + 1].reshape(1, -1, 3), 1.0)["sigma"]
            if ok(sig):
                break
            c *= 2
            assert c < 1e6
        norm[item] = trial[0]

    def empty_rays(dc, df):
        with torch.no_grad():
            return tr.render(ref32, norm, planes, o, d, dc, df)[3] == 0
    res = _render_case(dev, captured, rep, "opaque-and-empty", "dis", "fp32", norm, planes, o, d, opts, zero_depth_rays=empty_rays)
    empty = res["empty"]
    assert empty[2].all() and not empty[:2].any()
    rgb, seg, depth, wsum = res["out"]
    assert float((wsum[1].detach() - 1).abs().max()) < 1e-6              # item 1: all weight in front, nothing behind the opaque samples
    assert float(wsum[2].abs().max()) == 0.0
    all_depths = torch.cat([res["dc"], res["df"]], dim=2)
    assert torch.equal(depth[empty], torch.full_like(depth[empty], float(all_depths.max())))
    # the depth of an empty ray carries no gradient: a loss of those depths alone back-propagates to exact zeros
    leaves = (res["planes"], res["norm"], *res["dec"].parameters())
    for t in leaves:
        t.grad = None
    (depth[empty] * torch.randn_like(depth[empty])).sum().backward()
    for t in leaves:
        assert t.grad is None or (torch.isfinite(t.grad).all() and float(t.grad.abs().max()) == 0.0)


def _edge_points(n, m, h, w, box_warp, seed):
    """[n,m,3]: a third on texel centres (square planes: the same centre on all three planes), a sixth exactly on the
    faces +-box_warp/2, a sixth beyond them, the rest uniform over 1.3 x the box."""
    assert h == w
    gen = torch.Generator().manual_seed(seed)
    centres = ((2 * torch.arange(w, dtype=torch.float64) + 1) / w - 1) * box_warp / 2
    pts = (torch.rand(n, m, 3, generator=gen, dtype=torch.float64) * 2 - 1) * 0.65 * box_warp
    a, b, c = m // 3, m // 3 + m // 6, m // 3 + 2 * (m // 6)
    pts[:, :a] = centres[torch.randint(0, w, (n, a, 3), generator=gen)]
    face = pts[:, a:b].clone()
    axis = torch.randint(0, 3, (n, b - a), generator=gen)
    sign = torch.randint(0, 2, (n, b - a), generator=gen) * 2 - 1
    face.scatter_(2, axis.unsqueeze(-1), (sign * box_warp / 2).unsqueeze(-1).double())
    pts[:, a:b] = face
    out = pts[:, b:c].clone()
    out.scatter_(2, axis[:, :c - b].unsqueeze(-1), (sign[:, :c - b] * box_warp * (0.5 + 0.5 / w + 0.01)).unsqueeze(-1).double())
    pts[:, b:c] = out
    return pts.float()


RUN_MODEL_CASES = {"osg": ("fp32", 3), "dis": ("bf16x3", 1), "seg": ("bf16x3", 3)}     # (precision, plane batch)


@pytest.mark.parametrize("kind", list(RUN_MODEL_CASES))
def test_run_model_backward_edges(dev, record_property, kind):
    """run_model under autograd at points on texel centres, on and beyond the box faces; m = 2000 and m = 77 (fewer than one
    tile per item: the two-set path); the disentangled case reads one plane set [1,...] for all 3 point sets."""
    from nerffaceediting_b200.renderer import DisentangledImportanceRenderer, ImportanceRenderer
    rep = Report(record_property)
    precision, pb = RUN_MODEL_CASES[kind]
    dec = _decoder(kind, dev)
    ref_dec = tr.Decoder(dec, torch.float64, dev)
    norm, planes = _planes(407, pb, 16, 16, dev)
    box_warp = 1.6 if kind == "seg" else 1.0
    opts = dict(synth.FFHQ_RENDERING_OPTIONS, box_warp=box_warp, nfe_precision=precision)
    for m in (2000, 77):
        tag = f"run-model-edges-{kind} m={m}"
        coords = _edge_points(3, m, 16, 16, box_warp, 500 + m).to(dev)
        p_k, p_r = planes.detach().clone().requires_grad_(True), planes.detach().double().requires_grad_(True)
        n_k, n_r = norm.detach().clone().requires_grad_(True), norm.detach().double().requires_grad_(True)
        for p in (*dec.parameters(), *ref_dec.params.values()):
            p.grad = None
        if kind == "osg":
            out = ImportanceRenderer().run_model(p_k, dec, coords, torch.zeros_like(coords), opts)
        else:
            out = DisentangledImportanceRenderer().run_model(n_k, p_k, dec, coords, torch.zeros_like(coords), opts)
        want = tr.run_model(ref_dec, n_r, p_r, coords.double(), box_warp)
        assert set(out) == set(want)
        proj = dict(zip(("rgb", "sigma", "seg"), _projections([(3, m, 32), (3, m, 1), (3, m, 15)], 77 + m, dev)))
        for k in out:
            rep.rel(f"{tag} out.{k}", out[k], want[k], TOL[precision])
        sum((out[k].double() * proj[k]).sum() for k in out).backward()
        sum((want[k] * proj[k]).sum() for k in want).backward()
        leaves = [("g_planes", p_k, p_r, True)] + ([("g_norm", n_k, n_r, True)] if kind == "dis" else [])
        _compare_grads(rep, tag, precision, leaves, dec, ref_dec)


@pytest.mark.parametrize("swap", ["all", "one"])
def test_affine_chain_backward(dev, captured, record_property, swap):
    """raw -> normalize_plane -> denormalize_plane(norm, mean', std') -> renderer on the single-gather backward (bf16x3,
    23^2 rays x 16 samples per pass: tiles straddle the two items), against float64 autograd through (x - mean)/(std + 1e-8)
    and norm * std' + mean'.  The gradients of the raw planes, of mean' and of std' (one item's statistics broadcast over
    the batch when swap == 'one') are checked directly."""
    from nerffaceediting_b200 import ops, triplane
    from nerffaceediting_b200.renderer import DisentangledImportanceRenderer
    rep = Report(record_property)
    n, hw, res, s = 2, 32, 23, 16
    tag = f"affine-chain-{swap}"
    k_items = 1 if swap == "one" else n
    gen = torch.Generator().manual_seed(23)
    mean2 = (torch.randn(k_items, 96, 1, 1, generator=gen) * 0.5).to(dev)
    std2 = (torch.rand(k_items, 96, 1, 1, generator=gen) + 0.5).to(dev)
    raw0 = torch.from_numpy(synth.hash_normal(408, (n, 96, hw, hw)) * np.float32(1.5) - np.float32(0.3)).to(dev)
    o, d = _rays(n, res, dev)
    dec = _decoder("dis", dev)
    opts = dict(synth.FFHQ_RENDERING_OPTIONS, depth_resolution=s, depth_resolution_importance=s, nfe_deterministic=True,
                nfe_precision="bf16x3", nfe_single_gather=True)
    raw, m_k, s_k = (t.clone().requires_grad_(True) for t in (raw0, mean2, std2))
    norm, _, _ = triplane.normalize_plane(raw)
    planes = triplane.denormalize_plane(norm, m_k, s_k)
    captured.clear()
    ops.path_counts(reset=True)
    out = DisentangledImportanceRenderer()(norm.view(n, 3, 32, hw, hw), planes.view(n, 3, 32, hw, hw), dec, o, d, opts)
    assert ops.path_counts().get("render:training-single-gather", 0) == 1, ops.path_counts()
    dc, df = captured[0]
    ref_dec = tr.Decoder(dec, torch.float64, dev)
    x, m_r, s_r = (t.detach().double().requires_grad_(True) for t in (raw0, mean2, std2))
    mean, std = x.mean(dim=(-1, -2), keepdim=True), x.var(dim=(-1, -2), keepdim=True).sqrt()
    nrm = (x - mean) / (std + 1e-8)
    want = tr.render(ref_dec, nrm.view(n, 3, 32, hw, hw), (nrm * s_r + m_r).view(n, 3, 32, hw, hw), o, d, dc, df)
    proj = _projections([(n, res * res, 32), (n, res * res, 15), (n, res * res, 1), (n, res * res, 1)], 4343, dev)
    for nm, a, b in zip(("rgb", "seg", "depth", "wsum"), out, want):
        rep.rel(f"{tag} out.{nm}", a, b, 1e-4)
    sum((a.double() * w).sum() for a, w in zip(out, proj)).backward()
    sum((a * w).sum() for a, w in zip(want, proj)).backward()
    _compare_grads(rep, tag, "bf16x3", [("g_raw", raw, x, True), ("g_mean'", m_k, m_r, False), ("g_std'", s_k, s_r, False)],
                   dec, ref_dec)
