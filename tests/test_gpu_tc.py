"""GPU tests of the tensor path (AWB_PREC_F16: tcgen05 kind::f16 operands, fp32 accumulation in TMEM) against the
exact fp32 CUDA path and the CPU oracle.

Tolerances (single-pass fp16 operands == tf32-class, precision budget in DESIGN.md): loss rtol 2e-3;
gradients normwise 1e-2 per tensor; logits normwise 1e-3 and per-pixel 2e-2*max(1,|ref|); fitted masks
IoU >= 0.995 against the fp32 fit (north star: per-frame mIoU within 0.1 points)."""
import pytest
import torch

import __graft_entry__ as entry
from oracle import prior_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module", autouse=True)
def built():
    entry.build()


@pytest.fixture(scope="module")
def A():
    import awesome_b200
    return awesome_b200


def blob(H, W, seed=0, soft=True):
    g = torch.Generator().manual_seed(seed)
    yy, xx = torch.meshgrid(torch.linspace(0, 1, H), torch.linspace(0, 1, W), indexing="ij")
    sdf = torch.sqrt(((xx - 0.52) / 0.27) ** 2 + ((yy - 0.47) / 0.31) ** 2) - 1
    if soft:
        return torch.sigmoid((sdf + 0.05 * torch.randn(H, W, generator=g)) / 0.08)
    return (sdf > 0).float()


def pair(A, L, C=2, seed=0):
    torch.manual_seed(seed)
    m32 = A.ConvexNextNet(n_hidden_layers=L, in_features=C).to(DEV)
    m16 = A.ConvexNextNet(n_hidden_layers=L, in_features=C, precision="f16")
    m16.load_state_dict(m32.state_dict())
    return m32, m16.to(DEV)


def first_step_grads(fitter, P):
    """Adam after one step holds exp_avg = (1-beta1) * g: recover the reduced gradient from the optimizer state."""
    fitter.run(1)
    torch.cuda.synchronize()
    return fitter.opt_state[:4 * P].view(torch.float32).clone() * 10.0


@pytest.mark.parametrize("L,C,H,W", [(2, 2, 96, 128), (1, 2, 64, 100), (2, 3, 37, 53), (1, 3, 128, 148)])
def test_one_step_loss_and_gradients_vs_fp32(A, L, C, H, W):
    m32, m16 = pair(A, L, C)
    un = blob(H, W).to(DEV)
    if C == 2:
        grid = A.GridSpecHost("linspace", 1, H, W)
    else:
        grid = A.GridSpecHost("linspace", 1, H, W, t0=0.3, t_step=0.0)
    P = m32._arena.numel()
    f32 = m32.make_fitter(grid, un, A.LossConfig("mse"), A.OptimConfig("adam", lr=1e-3), use_graph=False)
    f16 = m16.make_fitter(grid, un, A.LossConfig("mse"), A.OptimConfig("adam", lr=1e-3), use_graph=False)
    g32 = first_step_grads(f32, P)
    g16 = first_step_grads(f16, P)
    l32, l16 = float(f32.scalars().last_loss), float(f16.scalars().last_loss)
    assert abs(l16 - l32) <= 2e-3 * abs(l32), (l16, l32)
    off = 0
    for name, p in m32.named_parameters():
        n = p.numel()
        a, b = g16[off:off + n], g32[off:off + n]
        rel = float((a - b).norm() / b.norm().clamp(min=1e-12))
        assert rel < 1e-2, f"{name}: normwise gradient error {rel:.3e}"
        off += n


def test_weighted_losses_on_tensor_path(A):
    m32, m16 = pair(A, 2)
    H, W = 80, 96
    hard = blob(H, W, soft=False).to(DEV)
    grid = A.GridSpecHost("index", 1, H, W)
    for loss in (A.LossConfig("fgbg_se", fg_weight=0.4), A.LossConfig("fgbg_bce_logits", fg_weight=0.3),
                 A.LossConfig("mse", mode="sssdms")):
        f32 = m32.make_fitter(grid, hard, loss, A.OptimConfig("adam", lr=0.0), use_graph=False)
        f16 = m16.make_fitter(grid, hard, loss, A.OptimConfig("adam", lr=0.0), use_graph=False)
        P = m32._arena.numel()
        g32, g16 = first_step_grads(f32, P), first_step_grads(f16, P)
        l32, l16 = float(f32.scalars().last_loss), float(f16.scalars().last_loss)
        assert abs(l16 - l32) <= 2e-3 * abs(l32), (loss, l16, l32)
        assert float((g16 - g32).norm() / g32.norm()) < 1e-2, loss


def test_tensor_forward_logits(A):
    m32, m16 = pair(A, 2)
    H, W = 120, 160
    un = blob(H, W).to(DEV)
    grid = A.GridSpecHost("linspace", 1, H, W)
    # train a while on the exact path so that logits are large and cancelling (worst case for fp16 operands)
    f32 = m32.make_fitter(grid, un, A.LossConfig("mse"), A.OptimConfig("adam", lr=1e-3), steps_per_graph=50)
    f32.run(600)
    m16.load_state_dict(m32.state_dict())
    m16.to(DEV)
    prior = m16._prior_for(torch.device(DEV))
    ws = prior.new_workspace(H * W, A._lib.AWB_WS_INFERENCE, DEV)
    y16 = prior.forward(m16._ensure_flat(), grid, A._lib.AWB_FWD_TC, ws)[0].reshape(-1)
    y32 = m32(grid.materialize(2, DEV)).reshape(-1)
    assert float((y16 - y32).norm() / y32.norm()) < 1e-3
    per_px = ((y16 - y32).abs() / y32.abs().clamp(min=1.0)).max()
    assert float(per_px) < 2e-2, float(per_px)
    flips = int(((y16 > 0) != (y32 > 0)).sum())
    assert flips <= max(3, H * W // 2000), flips


def test_fit_trajectory_and_mask_parity(A):
    """400 fused steps on both paths from the same init: final masks agree (IoU) and match the target equally well."""
    m32, m16 = pair(A, 2)
    H, W = 120, 160
    un = blob(H, W).to(DEV)
    grid = A.GridSpecHost("linspace", 1, H, W)
    hist = {}
    for name, m in (("fp32", m32), ("f16", m16)):
        f = m.make_fitter(grid, un, A.LossConfig("mse"), A.OptimConfig("adam", lr=1e-3), steps_per_graph=50)
        hist[name] = f.run(400).cpu().reshape(-1)
        f.raise_if_nonfinite()
    assert abs(float(hist["f16"][-1]) - float(hist["fp32"][-1])) < 0.1 * float(hist["fp32"][-1]) + 1e-4
    torch.testing.assert_close(hist["f16"][:20], hist["fp32"][:20], rtol=1e-2, atol=1e-5)
    y32 = m32(grid.materialize(2, DEV)).reshape(1, -1)
    y16 = m16(grid.materialize(2, DEV)).reshape(1, -1)          # exact forward of the f16-trained weights
    c = A.iou_counts(y16, y32, pred_is_logit=True)              # target arg thresholded at 0.5: use probabilities
    c = A.iou_counts(torch.sigmoid(y16), torch.sigmoid(y32), pred_is_logit=False).cpu()[0]
    iou_between = float(c[0]) / float(c[1] + c[2] - c[0])
    assert iou_between >= 0.995, iou_between
    ious = []
    for y in (y32, y16):
        c = A.iou_counts(torch.sigmoid(y), un.reshape(1, -1), pred_is_logit=False).cpu()[0]
        ious.append(float(c[0]) / float(c[1] + c[2] - c[0]))
    assert abs(ious[0] - ious[1]) <= 0.001, ious      # 0.1 IoU points
    for k in O.icnn_clamp_keys({k: v for k, v in m16.state_dict().items()}):
        assert float(m16.state_dict()[k].min()) >= 0.0


def test_frame_size_steps_vs_fp32_and_determinism(A):
    m32, m16 = pair(A, 2)
    H, W = 480, 640
    un = blob(H, W).to(DEV)
    grid = A.GridSpecHost("linspace", 1, H, W)
    f32 = m32.make_fitter(grid, un, A.LossConfig("mse"), A.OptimConfig("adam", lr=1e-3), use_graph=False)
    h32 = f32.run(10).cpu().reshape(-1)
    arena0 = m16._arena.clone()
    runs = []
    for _ in range(2):
        m16._arena.copy_(arena0)
        f16 = m16.make_fitter(grid, un, A.LossConfig("mse"), A.OptimConfig("adam", lr=1e-3), use_graph=False)
        runs.append((f16.run(10).cpu().reshape(-1), m16._arena.clone()))
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1]), "tensor path must be deterministic"
    torch.testing.assert_close(runs[0][0], h32, rtol=5e-3, atol=1e-6)


@pytest.mark.parametrize("kind", ["icnn", "flow3"])
def test_autograd_bridge_on_tensor_path(A, kind):
    """Joint / agent mode on the tensor path: loss.backward() through an f16 module re-runs the fused kernel with the
    upstream gradient (loss scale from the device-side max |dlogits|) -- gradients vs the exact fp32 module, for a
    mean-reduced and for a sum-reduced loss (six orders of magnitude apart in dlogits)."""
    torch.manual_seed(3)
    H, W = 72, 96
    if kind == "icnn":
        m32 = A.ConvexNextNet(n_hidden_layers=2).to(DEV)
        m16 = A.ConvexNextNet(n_hidden_layers=2, precision="f16")
        grid = A.GridSpecHost("linspace", 1, H, W).materialize(2, DEV)
    else:
        kw = dict(channels=3, hidden_units=32, flow_n_flows=6, flow_output_fn="tanh", convex_net_hidden_layers=2)
        m32 = A.real_nvp_path_connected_net(**kw).to(DEV)
        m16 = A.real_nvp_path_connected_net(precision="f16", **kw)
        grid = A.GridSpecHost("linspace", 2, H, W, t0=0.1, t_step=0.5).materialize(3, DEV)
        m32(grid)                                   # ActNorm data-dependent init, then copy
    m16.load_state_dict(m32.state_dict())
    m16 = m16.to(DEV)
    un = blob(H, W).to(DEV)
    for reduce in ("mean", "sum"):
        gs = {}
        for key, m in (("fp32", m32), ("f16", m16)):
            m.zero_grad()
            gin = grid.clone().requires_grad_(kind == "icnn")
            y = m(gin)
            l = (torch.sigmoid(y)[:, 0] - un) ** 2
            loss = l.mean() if reduce == "mean" else l.sum()
            loss.backward()
            gs[key] = (float(loss), torch.cat([p.grad.reshape(-1) for p in m.parameters()]),
                       gin.grad.clone() if kind == "icnn" else None)
        l32, g32, d32 = gs["fp32"]
        l16, g16, d16 = gs["f16"]
        assert abs(l16 - l32) <= 2e-3 * abs(l32), (reduce, l16, l32)
        rel = float((g16 - g32).norm() / g32.norm())
        assert rel < 2e-2, (kind, reduce, rel)
        if d32 is not None:
            assert float((d16 - d32).norm() / d32.norm()) < 2e-2
