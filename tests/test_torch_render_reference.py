"""Pins tests/_torch_render.py, the plain-torch restatement the backward edge tests compare the CUDA kernels with, to the
reference's own numbers on the CPU: the forward in float32 against render_small.npz and march.npz, and float64 autograd
gradients against backward.npz and run_model_bwd.npz.  A GPU test that disagrees with the restatement then points at a
kernel, not at the restatement.

Inputs are built as the GPU tests build them: rays from the oracle (bit-exact with the kernel), coarse depths from the
oracle's stratified sampler, fine depths from the oracle's full render (which matches render_small.npz, and whose resampler
is bit-exact with the GPU's on identical inputs)."""
import numpy as np
import pytest
import torch

import _torch_render as tr
import synth_inputs as synth
from oracle import nfe_oracle as orc
from _util import golden, oracle_decoder, rel_err
from test_oracle_golden import SMALL

TOL = 1e-4


def _module(g, prefix, kind, lr=1.0):
    """The package's decoder module with a golden state dict loaded (CPU)."""
    from nerffaceediting_b200.triplane import DisentangledOSGDecoder, OSGDecoder, SegmentationOSGDecoder
    cls = {"osg": OSGDecoder, "dis": DisentangledOSGDecoder, "seg": SegmentationOSGDecoder}[kind]
    dec = cls(32, {'decoder_lr_mul': lr, 'decoder_output_dim': 32, 'decoder_seg_dim': 15})
    dec.load_state_dict({k[len(prefix) + 1:]: torch.from_numpy(g[k]) for k in g.files
                         if k.startswith(prefix + ".") and k.split(".")[-1] in ("weight", "bias")})
    return dec


def _norm_of(raw):
    """triplane.py:56-65, the reference's own formula."""
    mean = raw.mean(dim=(-1, -2), keepdim=True)
    std = raw.var(dim=(-1, -2), keepdim=True).sqrt()
    return (raw - mean) / (std + 1e-8)


def _depths(g, tag, kind, opts, raw, norm, o, d, lr=1.0):
    """(coarse [N,R,S_c], fine [N,R,S_f] or None) exactly as the kernels would draw them in deterministic mode."""
    n, r, _ = o.shape
    s_c, s_f = opts['depth_resolution'], opts['depth_resolution_importance']
    if opts['ray_start'] == 'auto':
        t0, t1 = orc.ray_limits_box(o, d, opts['box_warp'])
        dc = orc.sample_stratified(n, r, s_c, start_per_ray=t0, end_per_ray=t1)
    elif opts['disparity_space_sampling']:
        dc = orc.sample_stratified(n, r, s_c, table=torch.linspace(0, 1, s_c).numpy(), ray_start=opts['ray_start'],
                                   ray_end=opts['ray_end'], disparity=True)
    else:
        dc = orc.sample_stratified(n, r, s_c, table=torch.linspace(opts['ray_start'], opts['ray_end'], s_c).numpy(),
                                   ray_start=opts['ray_start'], ray_end=opts['ray_end'])
    dc = dc.reshape(n, r, s_c)
    if not s_f:
        return dc, None
    k, a, b, cd, sd = oracle_decoder(g, f"{tag}.dec", kind, lr)
    st = orc.render(k, a, b, norm, raw, o, d, dc, torch.linspace(0, 1, s_f).numpy(), s_f, cd, sd, box_warp=opts['box_warp'],
                    white_back=opts['white_back'], return_stages=True)[4]
    return dc, st["depths_fine"]


@pytest.mark.parametrize("tag", list(SMALL))
def test_forward_float32_vs_render_small(tag):
    g = golden("render_small")
    kind, delta = SMALL[tag]
    opts = dict(synth.FFHQ_RENDERING_OPTIONS, **delta)
    lr = 0.5 if tag == "dis_lr05" else 1.0
    n, hw = 2, 16
    raw = synth.hash_normal(int(g[f"{tag}.seed"]), (n, 96, hw, hw)) * np.float32(1.5) - np.float32(0.3)
    norm = _norm_of(torch.from_numpy(raw)).numpy()
    o, d = orc.generate_rays(g["cam2world"], g["intrinsics"], 8)
    dc, df = _depths(g, tag, kind, opts, raw.reshape(n, 3, 32, hw, hw), None if kind == "osg" else norm.reshape(n, 3, 32, hw, hw), o, d, lr)
    dec = tr.Decoder(_module(g, f"{tag}.dec", kind, lr), torch.float32)
    with torch.no_grad():
        rgb, seg, depth, wsum = tr.render(dec, torch.from_numpy(norm).view(n, 3, 32, hw, hw), torch.from_numpy(raw).view(n, 3, 32, hw, hw),
                                          torch.from_numpy(o), torch.from_numpy(d), torch.from_numpy(dc),
                                          None if df is None else torch.from_numpy(df), opts['box_warp'], opts['white_back'])
    assert rel_err(rgb.numpy(), g[f"{tag}.rgb"]) < TOL
    assert rel_err(depth.numpy(), g[f"{tag}.depth"]) < TOL
    assert rel_err(wsum.numpy(), g[f"{tag}.wsum"]) < TOL
    if kind != "osg":
        assert rel_err(seg.numpy(), g[f"{tag}.seg"]) < TOL


def test_march_float32_vs_reference():
    g = golden("march")
    c, s, sg, dp = (torch.from_numpy(g[k]) for k in ("colors", "segs", "sigma", "depths"))
    for white, sfx in ((False, ""), (True, "_wb")):
        rgb, _, depth, w = tr.march(c, sg, dp, None, white)
        assert rel_err(rgb.numpy(), g[f"mip_rgb{sfx}"]) < 1e-6
        rgb, seg, depth_s, w_s = tr.march(c, sg, dp, s, white)
        assert rel_err(rgb.numpy(), g[f"seg_rgb{sfx}"]) < 1e-6
        assert rel_err(seg.numpy(), g[f"seg_seg{sfx}"]) < 1e-6
    assert rel_err(depth.numpy(), g["mip_depth"]) < 1e-6 and rel_err(w.numpy(), g["mip_weights"]) < 1e-6
    assert rel_err(depth_s.numpy(), g["seg_depth"]) < 1e-6 and rel_err(w_s.numpy(), g["seg_weights"]) < 1e-6
    assert depth_s[0, 0, 0] == dp.max()          # the zero-weight ray: NaN -> inf -> the global maximum depth


def test_march_behind_an_opaque_interval_vs_oracle():
    """Behind an interval with alpha == 1 exactly the transmittance is the reference's 1e-10 per such interval
    (ray_marcher.py: cumprod of 1 - alpha + 1e-10), not 0.  No golden has such an interval, so the weights behind it are
    compared element by element with the oracle's march (pinned to march.npz above), which restates the same term."""
    rng = np.random.default_rng(5)
    n, r, s = 1, 6, 16
    colors = rng.random((n, r, s, 32), dtype=np.float32)
    segs = rng.standard_normal((n, r, s, 15)).astype(np.float32)
    sigma = (rng.standard_normal((n, r, s, 1)) * 2 + 1).astype(np.float32)
    depths = (np.linspace(2.25, 3.3, s, dtype=np.float32)[None, None, :, None]
              + rng.random((n, r, s, 1)).astype(np.float32) * np.float32(0.02))
    sigma[0, :, 5] = 3000.0                        # intervals 4 and 5: alpha == 1 in float32
    rgb_o, seg_o, depth_o, w_o = orc.ray_march(colors, sigma, depths, segs)
    rgb, seg, depth, w = tr.march(*(torch.from_numpy(a) for a in (colors, sigma, depths, segs)))
    assert np.allclose(w_o[0, :, 5] / w_o[0, :, 4], 1e-10, rtol=1e-5)          # both intervals opaque
    behind = w_o[0, :, 6:, 0]
    assert (behind > 0).all() and (behind < 1e-15).all()
    assert float(np.max(np.abs(w.numpy()[0, :, 6:, 0] - behind) / behind)) < 1e-5
    assert rel_err(rgb.numpy(), rgb_o) < 1e-6 and rel_err(seg.numpy(), seg_o) < 1e-6 and rel_err(depth.numpy(), depth_o) < 1e-6


@pytest.mark.parametrize("tag", ["dis", "osg", "dis_wb"])
def test_float64_autograd_vs_backward_golden(tag):
    g = golden("backward")
    kind = "osg" if tag == "osg" else "dis"
    opts = dict(synth.FFHQ_RENDERING_OPTIONS, depth_resolution=12, depth_resolution_importance=12, white_back=tag == "dis_wb")
    n, hw = 2, 16
    raw = synth.hash_normal(300, (n, 96, hw, hw)) * np.float32(1.5) - np.float32(0.3)
    norm = g[f"{tag}.norm"] if kind == "dis" else None
    o, d = orc.generate_rays(g["cam2world"], g["intrinsics"], 8)
    dc, df = _depths(g, tag, kind, opts, raw.reshape(n, 3, 32, hw, hw), norm, o, d)
    dec = tr.Decoder(_module(g, f"{tag}.dec", kind), torch.float64)
    planes = torch.from_numpy(raw).double().view(n, 3, 32, hw, hw).requires_grad_(True)
    normt = torch.from_numpy(norm).double().requires_grad_(True) if norm is not None else None
    rgb, seg, depth, wsum = tr.render(dec, normt, planes, torch.from_numpy(o), torch.from_numpy(d), torch.from_numpy(dc), torch.from_numpy(df),
                                      opts['box_warp'], opts['white_back'])
    w = {k: torch.from_numpy(g[f"{tag}.{k}"]).double() for k in ("wr", "ws", "wd", "ww")}
    loss = (rgb * w["wr"]).sum() + (depth * w["wd"]).sum() + (wsum * w["ww"]).sum()
    if seg is not None:
        loss = loss + (seg * w["ws"]).sum()
    loss.backward()
    assert abs(float(loss.detach()) - float(g[f"{tag}.loss"])) <= TOL * max(1.0, abs(float(g[f"{tag}.loss"])))
    assert rel_err(planes.grad.numpy(), g[f"{tag}.g_planes"]) < TOL
    if normt is not None:
        assert rel_err(normt.grad.numpy(), g[f"{tag}.g_norm"]) < TOL
    for name, p in dec.params.items():
        assert rel_err(p.grad.numpy(), g[f"{tag}.g_dec.{name}"]) < TOL, name


def _check_decoder_grads(g, tag, dec, tol):
    """test_gpu_run_model_bwd._check_decoder_grads' rule: per parameter, max-norm error relative to that parameter's own
    gradient; a reference gradient that is pure cancellation noise (below 1e-4 of the largest) only has to be noise here too."""
    refs = {name: g[f"{tag}.g_dec.{name}"] for name in dec.params}
    top = max(float(np.abs(r).max()) for r in refs.values())
    for name, p in dec.params.items():
        ref = refs[name]
        if float(np.abs(ref).max()) < 1e-4 * top:
            assert p.grad is None or float(p.grad.abs().max()) < 1e-4 * top, name
            continue
        assert p.grad is not None and p.grad.shape == ref.shape, name
        assert rel_err(p.grad.numpy(), ref) < tol, name


@pytest.mark.parametrize("tag", ["dis_sigma", "dis_all", "dis_chain", "osg_all", "seg_all"])
def test_float64_autograd_vs_run_model_golden(tag):
    g = golden("run_model_bwd")
    kind = tag.split("_")[0]
    n, hw, m = 2, 16, 2000
    raw0 = torch.from_numpy(synth.hash_normal(310, (n, 96, hw, hw)) * np.float32(1.5) - np.float32(0.3)).double()
    dec = tr.Decoder(_module(g, f"{tag}.dec", kind), torch.float64)
    coords = torch.from_numpy(g["coords"]).double()
    if tag == "dis_chain":
        raw = raw0.clone().requires_grad_(True)
        norm, planes = _norm_of(raw).view(n, 3, 32, hw, hw), raw.view(n, 3, 32, hw, hw)
    else:
        norm = _norm_of(raw0).view(n, 3, 32, hw, hw).requires_grad_(True)
        planes = raw0.view(n, 3, 32, hw, hw).clone().requires_grad_(True)
    out = tr.run_model(dec, norm, planes, coords, 1.0)
    assert rel_err(out["sigma"].detach().numpy(), g[f"{tag}.out.sigma"]) < TOL
    if tag in ("dis_sigma", "dis_chain"):
        s = out["sigma"]
        loss = torch.nn.functional.l1_loss(s[:, :m // 2], s[:, m // 2:]) * 0.25
    else:
        loss = (out["rgb"] * torch.from_numpy(g["w_rgb"]).double()).sum() + (out["sigma"] * torch.from_numpy(g["w_sig"]).double()).sum()
        if "seg" in out:
            loss = loss + (out["seg"] * torch.from_numpy(g["w_seg"]).double()).sum()
    loss.backward()
    assert abs(float(loss.detach()) - float(g[f"{tag}.loss"])) <= TOL * max(1.0, abs(float(g[f"{tag}.loss"])))
    if tag == "dis_chain":
        assert rel_err(raw.grad.numpy(), g["dis_chain.g_raw"]) < TOL
    else:
        for t, key in ((planes, "g_planes"), (norm, "g_norm")):
            if f"{tag}.{key}" not in g:
                continue
            ref = g[f"{tag}.{key}"]
            got = t.grad.numpy() if t.grad is not None else np.zeros_like(ref)
            if np.any(ref):
                assert rel_err(got, ref) < TOL, key
            else:
                assert float(np.abs(got).max()) == 0.0, key
    _check_decoder_grads(g, tag, dec, TOL)

