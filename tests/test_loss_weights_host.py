"""Host side of the per-pixel loss weights (no GPU): the coefficients ``LossConfig.to_specs`` folds for weight maps and
an ignore label, checked by rebuilding the loss from the specs against the oracle, and the ``from_reference`` mapping of
the reference's weighted losses.  The device class counts are replaced by a CPU restatement of
``awb_target_counts_ignore``."""
import pytest
import torch

from oracle import prior_oracle as O

IGN = 2.0


@pytest.fixture()
def fit(monkeypatch):
    import awesome_b200.fit as F
    from awesome_b200 import _lib as L

    def counts(target, cls_rule, n_objects=1, ignore_value=None):
        t = target.reshape(n_objects, -1)
        keep = torch.ones_like(t, dtype=torch.bool) if ignore_value is None else t != ignore_value
        fg = (t < 0.5) if cls_rule == L.AWB_CLS_UNARY_LT_HALF else (t != 1.0)
        return torch.stack([(fg & keep).sum(1), (~fg & keep).sum(1)], 1).to(torch.int64)

    monkeypatch.setattr(F, "target_counts", counts)
    return F


def _target(N, O_=1, seed=0, frac=0.3, hard=False):
    g = torch.Generator().manual_seed(seed)
    t = torch.rand((O_, N), generator=g)
    if hard:
        t = (t >= 0.6).float()
    t = torch.where(torch.rand((O_, N), generator=g) < frac, torch.full_like(t, IGN), t)
    return t, 2.0 * torch.rand((O_, N), generator=g)


def _loss_from_specs(specs, t, w, y):
    """sum_n keep_n w_n coef(t_n) l(y_n, t_n), as the kernels compute it (float64)."""
    out = []
    for o, sp in enumerate(specs):
        to, yo = t[o].double(), y[o].double()
        fg = to < 0.5 if sp.cls_rule == 0 else to != 1.0
        coef = torch.where(fg, torch.tensor(sp.coef_fg, dtype=torch.float64), torch.tensor(sp.coef_bg, dtype=torch.float64))
        keep = (to != sp.ignore_value) if sp.ignore_enabled else torch.ones_like(fg)
        if sp.kind == 0:
            l = (to - torch.sigmoid(yo)) ** 2
        else:
            l = torch.nn.functional.binary_cross_entropy_with_logits(yo, to.clamp(0, 1), reduction="none")
        wo = w[o if w.shape[0] > 1 else 0].double() if w is not None else torch.ones_like(to)
        out.append(float(torch.where(keep, wo * coef * l, torch.zeros_like(l)).sum()))
    return out


@pytest.mark.parametrize("kind", ["mse", "bce"])
@pytest.mark.parametrize("mode", ["none", "ratio", "sssdms", "equal"])
def test_folded_coefficients_give_the_oracle_loss(fit, kind, mode):
    N, O_ = 4096, 2
    t, w = _target(N, O_, seed=1)
    y = torch.randn((O_, N), generator=torch.Generator().manual_seed(2))
    cfg = fit.LossConfig(kind, mode=mode, ratio=0.5, weight=w, ignore_value=IGN)
    wm = cfg.weight_map(O_, N, "cpu")
    specs = cfg.to_specs(t, wm)
    got = _loss_from_specs(specs, t, w, y)
    for o in range(O_):
        keep = t[o] != IGN
        tk = t[o][keep].double()
        cw = O.unaries_weight(tk, mode, 0.5)
        l = (tk - torch.sigmoid(y[o][keep].double())) ** 2 if kind == "mse" else \
            torch.nn.functional.binary_cross_entropy_with_logits(y[o][keep].double(), tk, reduction="none")
        ref = float((l * cw * w[o][keep].double()).sum() / keep.sum())
        assert got[o] == pytest.approx(ref, rel=1e-6), (o, got[o], ref)
        assert specs[o].ignore_enabled == 1 and specs[o].ignore_value == IGN
        assert specs[o].weight == wm[o].data_ptr()


def test_unweighted_specs_keep_their_coefficients(fit):
    """No map and no ignore label: the specs are those of the unweighted loss, with a zero tail."""
    t, _ = _target(1000, 1, frac=0.0)
    for cfg in (fit.LossConfig("mse"), fit.LossConfig("bce"), fit.LossConfig("mse", mode="sssdms")):
        sp = cfg.to_specs(t)[0]
        assert (sp.weight, sp.ignore_enabled, sp.ignore_value) == (None, 0, 0.0)
    sp = fit.LossConfig("mse").to_specs(t)[0]
    assert sp.coef_fg == pytest.approx(1.0 / 1000, rel=1e-7) and sp.coef_bg == sp.coef_fg


def test_weak_label_criterion_against_the_oracle(fit):
    """``WeightedLoss(BCELoss, "sssdms", noneclass=2)`` on {0, 1, 2} labels == ``loss_weighted_bce_sssdms``."""
    class BCELoss:
        pass

    class WeightedLoss:
        def __init__(self):
            self.criterion, self.mode, self.noneclass = BCELoss(), "sssdms", 2

    cfg = fit.LossConfig.from_reference(WeightedLoss())
    assert (cfg.kind, cfg.mode, cfg.ignore_value, cfg.weight) == ("bce", "sssdms", 2.0, None)
    t, _ = _target(5000, 1, seed=3, frac=0.9, hard=True)
    y = torch.randn((1, 5000), generator=torch.Generator().manual_seed(4))
    got = _loss_from_specs(cfg.to_specs(t), t, None, y)[0]
    ref = float(O.loss_weighted_bce_sssdms(torch.sigmoid(y.double()), t.double(), noneclass=2.0))
    assert got == pytest.approx(ref, rel=1e-6)


def test_from_reference_mapping(fit):
    class SE:
        pass

    class BCELoss:
        pass

    class UnariesWeightedLoss:
        def __init__(self, crit, mode, ratio=1.0):
            self.criterion, self.mode, self.ratio = crit, mode, ratio

    class WeightedLoss:
        def __init__(self, crit, mode, noneclass=None):
            self.criterion, self.mode, self.noneclass = crit, mode, noneclass

    m = fit.LossConfig.from_reference
    assert (m(UnariesWeightedLoss(BCELoss(), "ratio", 0.5)).kind, m(UnariesWeightedLoss(BCELoss(), "ratio", 0.5)).ratio) == \
        ("bce", 0.5)
    for mode in ("none", "ratio", "sssdms", "equal"):
        c = m(UnariesWeightedLoss(BCELoss(), mode))
        assert (c.kind, c.mode, c.ignore_value) == ("bce", mode, None)
        c = m(WeightedLoss(SE(), mode, noneclass=2))
        assert (c.kind, c.mode, c.ignore_value) == ("mse", mode, 2.0)
    assert m(WeightedLoss(BCELoss(), "none")).ignore_value is None
    assert m(UnariesWeightedLoss(SE(), "sssdms")).kind == "mse"

    class Focal:
        pass

    with pytest.raises(ValueError):
        m(WeightedLoss(Focal(), "none"))


def test_weight_map_shapes(fit):
    O_, B, H, W = 3, 2, 4, 5
    N = B * H * W
    cfg = fit.LossConfig("mse", weight=torch.rand(B, 1, H, W))
    assert cfg.weight_map(O_, N, "cpu").shape == (1, N)
    assert fit.LossConfig("mse", weight=torch.rand(O_, N)).weight_map(O_, N, "cpu").shape == (O_, N)
    assert fit.LossConfig("mse", weight=torch.rand(N).double()).weight_map(O_, N, "cpu").dtype == torch.float32
    with pytest.raises(ValueError):
        fit.LossConfig("mse", weight=torch.rand(N + 1)).weight_map(O_, N, "cpu")
    t, _ = _target(N, O_)
    w = fit.LossConfig("mse", weight=torch.rand(N)).weight_map(O_, N, "cpu")
    specs = fit.LossConfig("mse", weight=w).to_specs(t, w)
    assert {sp.weight for sp in specs} == {w.data_ptr()}          # one [N] map serves every object
