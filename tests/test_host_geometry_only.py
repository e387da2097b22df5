"""CPU-side tests of geometry-only renders (rendering_options['nfe_geometry_only']): the C ABI's workspace sizing and layout query,
the cfg struct, the render plan (which plane sets are staged, which path counter a call records) and the entry points that refuse
the option.  No kernel is launched here."""
import ctypes

import pytest
import torch

from nerffaceediting_b200 import _lib, ops


@pytest.fixture(scope="module")
def lib():
    from nerffaceediting_b200 import build
    build.build()
    return _lib.load()


def _cfg(kind, s_c, s_f, geometry):
    planes_cl = torch.empty(1, 3, 256, 256, 32, device="meta")
    cfg = ops.make_cfg(kind, planes_cl, s_c, s_f, 1.0, precision=_lib.PREC_BF16X3)
    cfg.geometry_only = int(geometry)
    return cfg


def _a256(x):
    return (x + 255) // 256 * 256


def test_cfg_appends_geometry_only_without_moving_fields():
    fields = [f[0] for f in _lib.NfeRenderCfg._fields_]
    assert fields[-1] == "geometry_only" and fields[-2] == "image_layout"
    assert _lib.NfeRenderCfg.geometry_only.offset == _lib.NfeRenderCfg.image_layout.offset + 4
    assert ops.make_cfg(ops.DEC_DISENTANGLED, torch.empty(1, 3, 8, 8, 32, device="meta"), 4, 4, 1.0).geometry_only == 0


@pytest.mark.parametrize("s_c,s_f", [(48, 48), (96, 96), (24, 0)])
def test_workspace_bytes_geometry_records_are_64_bytes(lib, s_c, s_f):
    """Records of a geometry-only render are {sigma, seg[15]}: 64 bytes per sample against 192, none for the OSG decoder."""
    n, rays = 4, 4096
    t = n * rays

    def expected(rec_bytes):
        b = _a256(64 * 4) + _a256(t * s_c * 4) + _a256(t * s_c * rec_bytes)
        if s_f:
            b += _a256(t * (s_c - 1) * 4) + 2 * _a256(t * s_f * 4) + _a256(t * s_f * rec_bytes)
        return b

    def ws(kind, geometry):
        return lib.nfe_render_workspace_bytes(ctypes.byref(_cfg(kind, s_c, s_f, geometry)), n, rays)
    for kind in (ops.DEC_DISENTANGLED, ops.DEC_SEGMENTATION):
        assert ws(kind, False) == expected(192)
        assert ws(kind, True) == expected(64)
        assert ws(kind, False) - ws(kind, True) == t * (s_c + s_f) * 128
    assert ws(ops.DEC_OSG, True) == expected(0)


def test_workspace_layout_rejects_geometry_only(lib):
    offs = (ctypes.c_int64 * 4)()
    assert lib.nfe_render_workspace_layout(ctypes.byref(_cfg(ops.DEC_DISENTANGLED, 48, 48, False)), 2, 64, offs) == 0
    assert lib.nfe_render_workspace_layout(ctypes.byref(_cfg(ops.DEC_DISENTANGLED, 48, 48, True)), 2, 64, offs) != 0
    assert b"geometry_only" in lib.nfe_last_error()


def test_field_plan_geometry_only(monkeypatch):
    """Disentangled decoder: only the normalised planes are staged, with or without provenance and in every precision; the call
    counts as render:geometry-only.  The OSG decoder stages its one plane set."""
    from nerffaceediting_b200 import plane_registry as reg
    from nerffaceediting_b200.renderer import field_plan
    reg.clear()
    monkeypatch.delenv("NFE_DEFAULT_PRECISION", raising=False)
    dis, osg = (ops.DEC_DISENTANGLED, None, None), (ops.DEC_OSG, None, None)
    norm, raw = torch.randn(2, 96, 4, 4), torch.randn(2, 96, 4, 4)
    reg.provenance_put(raw, norm, torch.full((2, 96), 2.0), torch.ones(2, 96))
    n5, r5, other = norm.view(2, 3, 32, 4, 4), raw.view(2, 3, 32, 4, 4), torch.randn(2, 3, 32, 4, 4)
    opts = dict(depth_resolution=48, depth_resolution_importance=48)
    for precision in ("fp32", "bf16x3", "bf16"):
        for pair in ((n5, r5), (n5, other)):
            p = field_plan("render", dis, *pair, dict(opts, nfe_precision=precision), 2, 64, False, geometry=True)
            assert p.geometry and p.affine is None and (p.stage_norm, p.stage_denorm) == (True, False)
            assert p.path == ("render", "geometry-only")
    p = field_plan("render", osg, None, r5, opts, 2, 64, False, geometry=True)
    assert p.geometry and (p.stage_norm, p.stage_denorm) == (False, True) and p.path == ("render", "geometry-only")
    assert not field_plan("render", dis, n5, r5, opts, 2, 64, False).geometry
    reg.clear()


def test_sharded_renderer_refuses_geometry_only():
    from nerffaceediting_b200.renderer import DisentangledImportanceRenderer
    from nerffaceediting_b200.sharding import ShardedRenderer, render_sharded
    opts = dict(nfe_geometry_only=True)
    o = torch.zeros(1, 4, 3)
    with pytest.raises(NotImplementedError, match="nfe_geometry_only"):
        render_sharded(DisentangledImportanceRenderer(), None, None, None, o, o, opts)
    with pytest.raises(NotImplementedError, match="nfe_geometry_only"):
        ShardedRenderer(DisentangledImportanceRenderer())(None, None, None, o, o, opts)
