"""The exact fp32 ICNN path at every width and depth class of ``WIDTH_CASES`` (``test_gpu_launch_regimes.py``), through the
two entry points that file does not run: the inference forward (``AWB_FWD_EXACT`` on an ``AWB_WS_INFERENCE`` workspace)
and the coordinate gradient of the module (``dgrid`` through ``awb_prior_backward``).

Rows wider than one k_gemm tile (ld > 144) are where the forward's skip / bias columns and the data gradient's skip
columns live in a second column tile; both must reach the logits and dgrid.  The references are the float64 oracle, with
the kink exclusion of ``test_gpu_coord_grad.py`` for dgrid, and the tolerances are those of the two files."""
import pytest
import torch

import __graft_entry__ as entry
from oracle import prior_oracle as O
from test_gpu_coord_grad import (CHUNK, KINK_MAX_FRACTION, TOL_DGRID, away_from_kinks, logits64, module_dgrid, p64, ref_dgrid,
                                 rows_of)
from test_gpu_launch_regimes import (TOL_FWD, WIDTH_CASES, check_regime, entry_err, grid_spec, make_handle, make_models,
                                     torch_grid)

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
# Excluded kink pixels of the depth-8 cases (L > 2 only; KINK_MAX_FRACTION = 5 % for the others): every pixel with one of
# L x h ReLU inputs within KINK of zero is left out, and 8 x 256 units put more pixels there.  Measured on one B200 at a
# 1000 W power limit: 9.9 % in c2-h256-L8, 6.8 % in c3-h200-L8.
KINK_MAX_FRACTION_DEEP = 0.15


@pytest.fixture(scope="module", autouse=True)
def built():
    entry.build()


@pytest.fixture(scope="module")
def A():
    import awesome_b200
    return awesome_b200


@pytest.mark.parametrize("case", WIDTH_CASES, ids=[c["id"] for c in WIDTH_CASES])
def test_inference_forward_against_float64(A, case):
    """Logits of the inference forward per entry against float64 within TOL_FWD, and bit for bit the logits of the training
    forward (the same kernels on a different workspace layout)."""
    r = check_regime(case)
    L = A._lib
    models = make_models(A, case)
    prior, params = make_handle(A, case, models)
    spec = grid_spec(A, case)
    N = spec.n_pixels
    logits, _ = prior.forward(params, spec, L.AWB_FWD_EXACT, prior.new_workspace(N, L.AWB_WS_INFERENCE, DEV))
    train, _ = prior.forward(params, spec, L.AWB_FWD_EXACT_TRAINING, prior.new_workspace(N, L.AWB_WS_TRAINING, DEV))
    assert torch.equal(logits, train)
    rows = O.pixelize(torch_grid("linspace", case["B"], case["H"], case["W"], case["C"]))
    worst = 0.0
    for o, m in enumerate(models):
        p = p64(m)
        with torch.no_grad():
            ref = torch.cat([logits64(case["kind"], p, rows[a:a + CHUNK].double()) for a in range(0, N, CHUNK)])
        worst = max(worst, entry_err(logits[o], ref))
    print(f"[exact width {case['id']}] N={N} ld={r['ld']}: inference logits {worst:.2e}")
    assert worst <= TOL_FWD, (case["id"], worst)


DGRID_CASES = [c for c in WIDTH_CASES if c["O"] == 1]


@pytest.mark.parametrize("case", DGRID_CASES, ids=[c["id"] for c in DGRID_CASES])
def test_module_dgrid_against_float64(A, case):
    """d sum(w * logits) / d grid through the module per entry against float64 autograd within TOL_DGRID, with w = 0 at the
    pixels within KINK of a ReLU kink (at most KINK_MAX_FRACTION of them, KINK_MAX_FRACTION_DEEP for L > 2)."""
    r = check_regime(case)
    m = make_models(A, case, seed=1)[0]
    B, C_, H, W = case["B"], case["C"], case["H"], case["W"]
    x4 = torch_grid("linspace", B, H, W, C_)
    torch.manual_seed(2)
    w, frac = away_from_kinks(case["kind"], m, rows_of(x4), torch.randn(B, 1, H, W, device=DEV),
                              max_fraction=KINK_MAX_FRACTION if case["L"] <= 2 else KINK_MAX_FRACTION_DEEP)
    dgrid = module_dgrid(m, x4, w)
    ref = ref_dgrid(case["kind"], m, rows_of(x4), w.reshape(-1))
    err = entry_err(rows_of(dgrid), ref)
    print(f"[exact width {case['id']}] N={r['N']} ld={r['ld']}: dgrid {err:.2e}  kink pixels {frac:.2%}")
    assert err <= TOL_DGRID, (case["id"], err)
