"""GPU parity tests of the ICNN prior-fit path: CUDA (through the C-ABI) vs golden fixtures produced
by the reference's modules, and vs the CPU oracle at FBMS frame size.

Tolerances (fp32 path): logits |err| <= 1e-4 * max(1,|ref|) (north-star bound is 1e-3); gradients
rtol 2e-3; post-step weights atol 2e-5; loss trajectories rtol 2e-4."""
import pytest
import torch

import __graft_entry__ as entry
from oracle import prior_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def built():
    entry.build()


@pytest.fixture(scope="module")
def A():
    import awesome_b200
    return awesome_b200


DEV = "cuda:0"


def logit_close(y, ref, tol=1e-4):
    err = (y - ref).abs() / ref.abs().clamp(min=1.0)
    assert float(err.max()) <= tol, f"max rel err {float(err.max()):.3e}"


def model_from(A, sd, L, **kw):
    m = A.ConvexNextNet(n_hidden_layers=L, **kw)
    m.load_state_dict(sd)
    return m.to(DEV)


def test_forward_matches_reference_c1_c2(A, golden):
    g = golden("icnn_c1.pt")
    m = model_from(A, g["init"], 1)
    logit_close(m(g["grid"].to(DEV)).cpu(), g["logits0"])
    m.load_state_dict(g["after6"])
    logit_close(m(g["grid"].to(DEV)).cpu(), g["logits6"])
    g2 = golden("icnn_c2.pt")
    m2 = model_from(A, g2["init"], 2)
    logit_close(m2(g2["grid"].to(DEV)).cpu(), g2["logits0"])
    # pixel-row input [N,C] -> [N,1] (pixelize() pass-through, awesome/util/pixelize.py:23-28)
    rows = O.pixelize(g2["grid"]).to(DEV)
    logit_close(m2(rows).cpu(), O.pixelize(g2["logits0"]))
    cn = A.ConvexNet()
    cn.load_state_dict(g2["convexnet_init"])
    logit_close(cn.to(DEV)(rows).cpu(), g2["convexnet_logits"])


def test_generated_grids_equal_explicit(A, golden):
    g2 = golden("icnn_c2.pt")
    m = model_from(A, g2["init"], 2)
    H, W = g2["H"], g2["W"]
    prior = m._prior_for(torch.device(DEV))
    ws = prior.new_workspace(H * W, A._lib.AWB_WS_INFERENCE, DEV)
    y_gen, _ = prior.forward(m._ensure_flat(), A.GridSpecHost("linspace", 1, H, W), A._lib.AWB_FWD_EXACT, ws)
    y_exp = m(g2["grid"].to(DEV)).reshape(1, -1)
    assert torch.equal(y_gen, y_exp), "in-kernel linspace grid differs from torch.linspace"
    g1 = golden("icnn_c1.pt")
    m1 = model_from(A, g1["init"], 1)
    H, W = g1["H"], g1["W"]
    prior = m1._prior_for(torch.device(DEV))
    ws = prior.new_workspace(H * W, A._lib.AWB_WS_INFERENCE, DEV)
    y_gen, _ = prior.forward(m1._ensure_flat(), A.GridSpecHost("index", 1, H, W), A._lib.AWB_FWD_EXACT, ws)
    assert torch.equal(y_gen, m1(g1["grid"].to(DEV)).reshape(1, -1))


def test_autograd_backward_matches_reference_grads(A, golden):
    g = golden("icnn_c2.pt")
    m = model_from(A, g["init"], 2)
    un = g["unaries"].to(DEV)
    for mode in ("none", "sssdms"):
        m.zero_grad()
        y = m(g["grid"].to(DEV))
        loss = O.loss_unaries_weighted_se(y, un, mode)          # torch ops on the device, autograd into our kernels
        loss.backward()
        torch.testing.assert_close(loss.detach().cpu(), g[f"loss_{mode}"], rtol=1e-5, atol=1e-7)
        for k, p in m.named_parameters():
            torch.testing.assert_close(p.grad.cpu(), g[f"grads_{mode}"][k], rtol=2e-3, atol=2e-8, msg=lambda s: f"{k}: {s}")


def test_input_gradient(A, golden):
    """model_input_requires_grad configs (gradient penalty): d logits / d grid."""
    g = golden("icnn_c2.pt")
    m = model_from(A, g["init"], 2)
    x = g["grid"].to(DEV).clone().requires_grad_(True)
    m(x).sum().backward()
    p = O.clone_params(g["init"])
    xr = O.pixelize(g["grid"]).clone().requires_grad_(True)
    O.icnn_forward(p, xr).sum().backward()
    torch.testing.assert_close(O.pixelize(x.grad.cpu()), xr.grad, rtol=1e-3, atol=1e-6)


def test_fused_fit_c1_trajectory(A, golden):
    """Config 1: fg/bg-weighted SE, Adam lr 2e-3, clamp -- six fused steps vs the reference loop."""
    g = golden("icnn_c1.pt")
    for use_graph in (False, True):
        m = model_from(A, g["init"], 1)
        fitter = m.make_fitter(A.GridSpecHost("index", 1, g["H"], g["W"]), g["unaries"].to(DEV),
                               A.LossConfig("fgbg_se", fg_weight=0.4), A.OptimConfig("adam", lr=2e-3),
                               steps_per_graph=3, use_graph=use_graph)
        h1 = fitter.run(1)
        for k, v in m.state_dict().items():
            torch.testing.assert_close(v.cpu(), g["after1"][k], rtol=1e-4, atol=2e-6, msg=lambda s: f"{k}: {s}")
        h5 = fitter.run(5)
        hist = torch.cat([h1, h5]).cpu().reshape(-1)
        torch.testing.assert_close(hist, g["loss_hist"], rtol=2e-4, atol=1e-7)
        for k, v in m.state_dict().items():
            torch.testing.assert_close(v.cpu(), g["after6"][k], rtol=1e-3, atol=2e-5, msg=lambda s: f"{k}: {s}")
        for k in O.icnn_clamp_keys(g["init"]):
            assert float(m.state_dict()[k].min()) >= 0.0
        assert fitter.scalars().step == 6 and fitter.scalars().nonfinite == 0


def test_fused_fit_c2_adam_and_adamax_plateau(A, golden):
    g = golden("icnn_c2.pt")
    m = model_from(A, g["init"], 2)
    fitter = m.make_fitter(g["grid"].to(DEV), g["unaries"].to(DEV), A.LossConfig("mse"),
                           A.OptimConfig("adam", lr=1e-3), use_graph=False)
    hist = fitter.run(4).cpu().reshape(-1)
    torch.testing.assert_close(hist, g["adam_hist"], rtol=2e-4, atol=1e-7)
    for k, v in m.state_dict().items():
        torch.testing.assert_close(v.cpu(), g["adam_after4"][k], rtol=1e-3, atol=2e-5, msg=lambda s: f"{k}: {s}")
    m = model_from(A, g["init"], 2)
    pa = g["plateau_args"]
    fitter = m.make_fitter(g["grid"].to(DEV), g["unaries"].to(DEV), A.LossConfig("mse"),
                           A.OptimConfig("adamax", lr=1e-3, plateau=True, patience=pa["patience"],
                                         factor=pa["factor"], threshold=pa["threshold"]), use_graph=False)
    lrs, hist = [], []
    for _ in range(8):
        hist.append(float(fitter.run(1).cpu()))
        lrs.append(fitter.scalars().lr[1])
    torch.testing.assert_close(torch.tensor(hist), g["adamax_hist"], rtol=2e-4, atol=1e-7)
    torch.testing.assert_close(torch.tensor(lrs, dtype=torch.float64), g["adamax_lrs"].double(), rtol=1e-6, atol=0)
    for k, v in m.state_dict().items():
        torch.testing.assert_close(v.cpu(), g["adamax_after8"][k], rtol=1e-3, atol=2e-5, msg=lambda s: f"{k}: {s}")


@pytest.mark.parametrize("mode", ["ratio", "sssdms", "equal"])
def test_fused_weighted_loss_modes(A, golden, mode):
    g = golden("icnn_c2.pt")
    m = model_from(A, g["init"], 2)
    fitter = m.make_fitter(g["grid"].to(DEV), g["unaries"].to(DEV), A.LossConfig("mse", mode=mode, ratio=0.5),
                           A.OptimConfig("adam", lr=0.0), use_graph=False)
    loss = fitter.run(1).cpu().reshape(())
    torch.testing.assert_close(loss, g[f"loss_{mode}"], rtol=1e-5, atol=1e-7)


def test_fbms_frame_size_vs_oracle(A):
    """640x480 (BASELINE config 2 frame): forward + 2 fused steps vs the CPU oracle; clamp idempotence;
    deterministic replays."""
    torch.manual_seed(42)
    H, W = 480, 640
    m = A.ConvexNextNet(n_hidden_layers=2).to(DEV)
    p = {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}
    yy, xx = torch.meshgrid(torch.linspace(0, 1, H), torch.linspace(0, 1, W), indexing="ij")
    un = torch.sigmoid((torch.sqrt(((xx - 0.45) / 0.3) ** 2 + ((yy - 0.55) / 0.2) ** 2) - 1) / 0.08)
    rows = O.pixelize(O.grid_linspace(H, W)[None])
    ref = O.icnn_forward(p, rows)
    y = m(O.grid_linspace(H, W)[None].to(DEV)).cpu()
    logit_close(O.pixelize(y), ref)
    arena0 = m._arena.clone()
    runs = []
    for _ in range(2):
        m._arena.copy_(arena0)
        fitter = m.make_fitter(A.GridSpecHost("linspace", 1, H, W), un.to(DEV), A.LossConfig("mse"),
                               A.OptimConfig("adam", lr=1e-3), use_graph=False)
        runs.append((fitter.run(2).cpu().reshape(-1), m._arena.clone()))
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1]), "fit is not deterministic"
    rec = []
    O.fit_icnn(p, rows, un, steps=2, optimizer="adam", lr=1e-3, record=rec)
    torch.testing.assert_close(runs[0][0], torch.tensor(rec), rtol=2e-4, atol=1e-7)
    for k, v in m.state_dict().items():
        torch.testing.assert_close(v.cpu(), p[k], rtol=1e-3, atol=2e-5, msg=lambda s: f"{k}: {s}")
    before = m._arena.clone()
    m.enforce_convexity()
    assert torch.equal(before, m._arena), "clamp must be idempotent after a fused step"


def test_ragged_and_tiny_sizes(A, golden):
    g = golden("icnn_c2.pt")
    m = model_from(A, g["init"], 2)
    p = O.clone_params(g["init"])
    for (H, W) in [(1, 1), (3, 5), (17, 129), (1, 300)]:
        grid = torch.rand(1, 2, H, W)
        logit_close(m(grid.to(DEV)).cpu(), O.unpixelize(O.icnn_forward(p, O.pixelize(grid)), 1, H, W))
    with pytest.raises(ValueError):
        m(torch.zeros(1, 3, 4, 4, device=DEV))


def test_nonfinite_loss_is_flagged_not_trapped(A, golden):
    g = golden("icnn_c2.pt")
    m = model_from(A, g["init"], 2)
    un = g["unaries"].clone()
    un[0, 0, 0, 0] = float("nan")
    fitter = m.make_fitter(g["grid"].to(DEV), un.to(DEV), A.LossConfig("mse"), A.OptimConfig("adam"), use_graph=False)
    before = m._arena.clone()
    fitter.run(1)
    assert fitter.scalars().nonfinite == 1
    assert torch.equal(before, m._arena), "a non-finite loss must not touch the parameters"
    with pytest.raises(ValueError, match="Loss is nan or inf"):
        fitter.raise_if_nonfinite()


def test_iou_and_target_counts(A, golden):
    g = golden("losses.pt")
    a, b = g["miou_a"], g["miou_b"]
    c = A.iou_counts(a.to(DEV), b.to(DEV), pred_is_logit=False).cpu()[0]
    iou = float(c[0]) / float(c[1] + c[2] - c[0])
    assert abs(iou - float(g["miou_ab"])) < 1e-6
    assert abs(iou - O.miou_binary_inverted(a, b)) < 1e-9
    t = golden("icnn_c2.pt")["unaries"]
    cnt = A.target_counts(t.to(DEV), 0).cpu()[0]
    assert int(cnt[0]) == int((t < 0.5).sum()) and int(cnt[1]) == int((t >= 0.5).sum())
