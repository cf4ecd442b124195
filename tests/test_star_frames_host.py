"""Whole-frame fits of the star-shape prior, host side (no GPU): the notebook's grid, ``make_fitter`` routing,
``reset_parameters`` in the arena, the forward's grid handling and the C-ABI prototypes it relies on."""
import ctypes as C

import pytest
import torch

import awesome_b200 as A
from awesome_b200 import _lib as L
from awesome_b200 import fit as F
from awesome_b200 import synth
from awesome_b200.model import star_net as S


def test_create_grid_matches_fit_likelihood_coordinates():
    """``fit_likelihood`` samples pixel (i, j) at ``(i / (H - 1) - 0.5, j / (W - 1) - 0.5)``: the grid holds exactly
    those values, channel 0 the row and channel 1 the column."""
    H, W = 37, 53
    lk = synth.star_unaries(H, W, seed=3)
    g = A.StarShapedNet.create_grid(H, W, B=2)
    assert g.shape == (2, 2, H, W) and g.dtype == torch.float32 and g.is_contiguous()
    for mask in (lk < 0.5, lk > 0.5):
        idx = torch.nonzero(mask)
        pix = torch.stack([idx[:, 0] / (H - 1) - 0.5, idx[:, 1] / (W - 1) - 0.5], dim=1).float()   # fit_likelihood
        rows = g[1].permute(1, 2, 0)[mask]
        assert torch.equal(rows, pix)
    with pytest.raises(ValueError):
        A.StarShapedNet.create_grid(1, 8)


def test_star_unaries_are_a_non_convex_star():
    u = synth.star_unaries(96, 128, seed=1)
    assert u.shape == (96, 128) and float(u.min()) >= 0 and float(u.max()) <= 1
    fg = u < 0.5
    assert 0.05 < float(fg.float().mean()) < 0.5
    # the centre is inside, and the blob is not convex: some midpoint of two fg pixels is bg
    assert bool(fg[48, 64])
    ij = torch.nonzero(fg).float()
    g = torch.Generator().manual_seed(0)
    a, b = ij[torch.randint(len(ij), (4000,), generator=g)], ij[torch.randint(len(ij), (4000,), generator=g)]
    mid = ((a + b) / 2).round().long()
    assert not bool(fg[mid[:, 0], mid[:, 1]].all())
    assert torch.equal(u, synth.star_unaries(96, 128, seed=1))


class _Recorder:
    def __init__(self, *args, **kw):
        self.args, self.kw = args, kw


def test_make_fitter_routes_grids_to_prior_fitter(monkeypatch):
    torch.manual_seed(0)
    m = A.StarShapedNet(16)
    monkeypatch.setattr(m, "_prior_for", lambda device: "handle")
    monkeypatch.setattr(F, "PriorFitter", _Recorder)
    monkeypatch.setattr(S, "StarFitter", _Recorder)
    grid = A.StarShapedNet.create_grid(6, 7)
    target = torch.rand(42)
    f = m.make_fitter(grid, target, A.LossConfig("bce"), A.OptimConfig("adam", lr=1e-2), steps_per_graph=5)
    prior, arena, spec, tgt, loss, optim = f.args
    assert prior == "handle" and arena.data_ptr() == m._arena.data_ptr()
    assert spec.mode == "explicit" and (spec.B, spec.H, spec.W) == (1, 6, 7) and torch.equal(spec.grid, grid)
    assert tgt is target and loss.kind == "bce" and optim.lr == 1e-2
    assert f.kw == dict(active_groups=0b010, steps_per_graph=5)         # the offset starts frozen
    m.offset.requires_grad_(True)
    f = m.make_fitter(grid, target)
    assert f.kw["active_groups"] == 0b110 and f.args[4].kind == "mse"
    # a generated grid is materialised (GridSpecHost's own convention)
    gs = A.GridSpecHost("linspace", 1, 6, 7)
    f = m.make_fitter(gs, target)
    assert f.args[2].mode == "explicit" and torch.equal(f.args[2].grid, gs.materialize(2, "cpu"))
    with pytest.raises(ValueError):
        m.make_fitter(grid)
    # no grid: the notebook's sampled-point fitter, with the old keyword calls
    f = m.make_fitter()
    assert f.args == (m, None, None)
    opt, loss = A.OptimConfig("adam", lr=0.0), A.LossConfig("mse")
    f = m.make_fitter(optim=opt, loss=loss)
    assert f.args == (m, opt, loss)


def test_reset_parameters_redraws_in_place_in_the_arena():
    torch.manual_seed(5)
    m = A.StarShapedNet(24)
    first = {k: v.clone() for k, v in m.state_dict().items()}
    arena = m._ensure_flat()
    ptrs = {k: p.data_ptr() for k, p in m.named_parameters()}
    with torch.no_grad():
        m.offset.fill_(0.25)
        arena.add_(1.0)
    m.offset.requires_grad_(True)
    torch.manual_seed(5)
    torch.zeros(1, 2)            # the constructor's offset draws nothing: the weights follow the same stream
    m.reset_parameters()
    assert m._ensure_flat().data_ptr() == arena.data_ptr()
    assert {k: p.data_ptr() for k, p in m.named_parameters()} == ptrs
    for k, v in m.state_dict().items():
        assert torch.equal(v, first[k]), k                    # the constructor's draw, offset back to 0
    assert m.offset.requires_grad
    assert torch.equal(arena, torch.cat([v.reshape(-1) for v in first.values()]))


def test_forward_rejects_bad_shapes_and_cpu_inputs():
    m = A.StarShapedNet(8)
    for bad in (torch.zeros(5, 3), torch.zeros(1, 3, 4, 4), torch.zeros(2, 2, 2, 2, 2)):
        with pytest.raises(ValueError):
            m(bad)
    with pytest.raises(L.AwbLibraryError):
        m(torch.zeros(1, 2, 4, 4))


def test_prototypes_of_the_fit_entry_points():
    """The star grid fit goes through the generic fit entry points; their ctypes prototypes take a grid spec and one
    loss spec per object (with the weight / ignore tail) and the workspace query takes a layout."""
    sym = {name: (res, args) for name, res, args in L.SYMBOLS}
    for name in ("awb_prior_fit_step", "awb_prior_fit_steps", "awb_prior_fit_host_frames"):
        res, args = sym[name]
        assert res is C.c_int and args[3] == C.POINTER(L.GridSpec) and C.POINTER(L.LossSpec) in args
    assert sym["awb_prior_workspace_bytes"] == (C.c_int64, [C.c_void_p, C.c_int64, C.c_int32])
    assert [f[0] for f in L.LossSpec._fields_][-3:] == ["weight", "ignore_enabled", "ignore_value"]
    assert L.AWB_WS_FIT_STEP == 2 and L.AWB_KIND_STAR == 2
