"""Full-schedule parity at BASELINE sizes: the device fits (exact fp32 path AND the tcgen05 tensor path) against fits the
REFERENCE's own modules ran to completion on the CPU (``tests/golden/make_golden_full.py`` -> ``full_*.pt``).

North-star criterion (iii): per-frame mIoU within 0.1 points of the reference.  Trajectories of 2 000 - 4 000 optimizer
steps are not comparable bit for bit between a CPU and a GPU (summation order), fitted masks are: every test compares
``MIOU(average="binary", invert=True)`` (``awesome/measures/miou.py:29-48``) of the fitted mask against the target between
the device fit and the reference fit (tolerance 0.1 points = 1e-3), and reports the direct IoU between the two masks.
The inputs are regenerated from seeds by ``awesome_b200/synth.py`` and checked against the fixture's checksum."""
import os

import pytest
import torch

import __graft_entry__ as entry
from awesome_b200 import synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
MIOU_TOL = 1e-3          # 0.1 points
TC_LOGIT_BOUND = 3e-2    # stated per-pixel bound of tensor-path logits, |d| / max(1, |y|) (include/awb.h, DESIGN 5); measured 2.2e-2


@pytest.fixture(scope="module", autouse=True)
def built():
    entry.build()


@pytest.fixture(scope="module")
def A():
    import awesome_b200
    return awesome_b200


def _check_inputs(unaries, chk):
    assert list(unaries.shape) == chk["shape"] or list(unaries.shape) == chk["shape"][-2:]
    assert abs(float(unaries.double().mean()) - chk["mean"]) < 1e-6
    assert abs(int((unaries < 0.5).sum()) - chk["fg"]) <= 2      # soft unaries: a last-ulp sigmoid may move a pixel


TRACE_LAST, TRACE_EVERY = 200, 10      # make_golden_full.py: IoU before steps n-200, n-190, ..., n-10 and after step n


def _run_traced(fitter, model, grid, target_fg, steps):
    """``steps`` fused fit steps; like the fixture, the IoU of the current mask is sampled every 10 steps over the last
    200 (the fits end without a learning-rate decay: one particular step's mask moves by tenths of a point)."""
    head = steps - TRACE_LAST
    hist = [fitter.run(head)]
    trace = []
    for _ in range(TRACE_LAST // TRACE_EVERY):
        trace.append(synth.fg_iou(_fitted_fg(model, grid), target_fg))
        hist.append(fitter.run(TRACE_EVERY))
    trace.append(synth.fg_iou(_fitted_fg(model, grid), target_fg))
    return torch.cat(hist).reshape(-1).cpu(), torch.tensor(trace)


def _compare_trace(name, trace, ref_trace, replicas=None):
    """Median mIoU over the last 200 steps within 0.1 points of the reference's.  Where the fixture holds REPLICAS of the
    reference fit (the reference's own modules, same schedule, parameters perturbed by one part in 10^7: the fit is chaotic
    at the level of an fp32 rounding, see ``make_golden_full.py:gen_c3nb_replicas``), the reference is the band its own
    runs span, not one trajectory."""
    med = float(trace.median())
    ref_meds = [float(ref_trace.median())] + ([float(r.median()) for r in replicas] if replicas is not None else [])
    lo, hi = min(ref_meds), max(ref_meds)
    ref_txt = f"{100 * lo:.3f}" if len(ref_meds) == 1 else f"{100 * lo:.3f}..{100 * hi:.3f} over {len(ref_meds)} runs"
    delta = med - hi if med > hi else (med - lo if med < lo else 0.0)
    print(f"[{name}] median mIoU over the last {TRACE_LAST} steps: device {100 * med:.3f}  reference {ref_txt}  "
          f"(delta {100 * delta:+.3f} points); step-to-step spread: device {100 * float(trace.min()):.2f}.."
          f"{100 * float(trace.max()):.2f}, reference {100 * float(ref_trace.min()):.2f}..{100 * float(ref_trace.max()):.2f}")
    assert abs(delta) <= MIOU_TOL, (name, med, ref_meds)


def _fitted_fg(model, grid):
    with torch.no_grad():
        return (torch.sigmoid(model(grid)) < 0.5).reshape(grid.shape[-2:]).cpu()


def _compare(name, fg, ref_fg, target_fg, ref_iou=None):
    iou_ours, iou_ref = synth.fg_iou(fg, target_fg), synth.fg_iou(ref_fg, target_fg)
    direct = synth.fg_iou(fg, ref_fg)
    print(f"[{name}] mIoU vs target: device {100 * iou_ours:.3f}  reference {100 * iou_ref:.3f}  "
          f"(delta {100 * (iou_ours - iou_ref):+.3f} points); IoU(device mask, reference mask) {100 * direct:.3f}")
    if ref_iou is not None:
        assert abs(iou_ref - ref_iou) < 1e-6      # the fixture's own record of the reference's IoU
    assert abs(iou_ours - iou_ref) <= MIOU_TOL, (name, iou_ours, iou_ref)
    return direct


@pytest.mark.parametrize("precision", ["fp32", "f16"])
def test_c1_convexity_notebook_2000_steps(A, golden, precision):
    """BASELINE configs[0]: 256x256, ConvexNextNet(L=1), notebook grid, fg/bg-weighted SE (0.4), Adam 2e-3, 2000 steps."""
    g = golden("full_c1.pt")
    H, W = g["H"], g["W"]
    un = synth.c1_unaries(H, W, seed=0)
    _check_inputs(un, g["unaries_check"])
    m = A.ConvexNextNet(n_hidden_layers=1, precision=precision)
    m.load_state_dict(g["init"])
    m = m.to(DEV)
    spec = A.GridSpecHost("index", 1, H, W)
    f = m.make_fitter(spec, un.to(DEV), A.LossConfig("fgbg_se", fg_weight=0.4), A.OptimConfig("adam", lr=2e-3))
    x = spec.materialize(2, DEV)
    hist, trace = _run_traced(f, m, x, un < 0.5, 2000)
    f.raise_if_nonfinite()
    # the first steps are comparable one by one, the end of the curve in value
    torch.testing.assert_close(hist[:3], g["loss_hist"][:3], rtol=5e-3 if precision == "f16" else 1e-4, atol=1e-7)
    assert abs(float(hist[-50:].mean()) - float(g["loss_hist"][-50:].mean())) < 0.02 * float(g["loss_hist"][-50:].mean())
    _compare_trace(f"c1 {precision}", trace, g["iou_trace"])
    fg = _fitted_fg(m, x)
    ref_fg = synth.unpack_mask(g["mask_fg_packed"], H, W)
    direct = _compare(f"c1 {precision}", fg, ref_fg, un < 0.5, g["iou_vs_unaries"])
    assert direct > 0.99
    # the convex shape under the noise is what the prior is for
    clean = synth.c1_clean_mask(H, W, 0) < 0.5
    assert abs(synth.fg_iou(fg, clean) - g["iou_vs_clean"]) <= MIOU_TOL


def _c3nb_model(A, g, precision, state):
    H, W = g["H"], g["W"]
    fl = g["schedule"]["flow"]
    flow = A.init_realnvp(channels=2, n_flows=fl["n_flows"], hidden_units=fl["hidden_units"], height=H, width=W,
                          output_fn=fl["output_fn"])
    norm = A.get_norm("minmax", dim=(0, 2, 3))
    norm.fit(A.GridSpecHost("index", 1, H, W).materialize(2, "cpu"))
    m = A.PathConnectedNet(convex_net=A.ConvexNextNet(n_hidden_layers=2, precision=precision),
                           flow_net=A.NormNet(net=A.PixelizeNet(flow), norm=norm))
    m.load_state_dict(g[state])
    return m.to(DEV)


@pytest.mark.parametrize("precision", ["fp32", "f16"])
def test_c3_path_connectedness_notebook_2000_steps(A, golden, precision):
    """BASELINE configs[2], notebook variant: 320x213, RealNVP(m=8, F=10, tanh) o ConvexNextNet(L=2), Adamax (flow lr 2e-3,
    wd 1e-5; rest 1e-3), fg/bg-weighted BCE-with-logits (0.3), 2000 steps from the reference's flow-identity state."""
    g = golden("full_c3nb.pt")
    H, W = g["H"], g["W"]
    un = synth.c3_unaries(H, W, seed=7, hard=True)
    _check_inputs(un, g["unaries_check"])
    m = _c3nb_model(A, g, precision, "after_identity")
    spec = A.GridSpecHost("index", 1, H, W)
    opt = A.OptimConfig("adamax", lr=[2e-3, 1e-3, 1e-3, 1e-3], weight_decay=[1e-5, 0.0, 0.0, 0.0])
    f = m.make_fitter(spec, un.to(DEV), A.LossConfig("fgbg_bce_logits", fg_weight=0.3), opt)
    x = spec.materialize(2, DEV)
    hist, trace = _run_traced(f, m, x, un < 0.5, 2000)
    f.raise_if_nonfinite()
    torch.testing.assert_close(hist[:3], g["loss_hist"][:3], rtol=5e-3 if precision == "f16" else 2e-4, atol=1e-7)
    # This fit (Adamax at a constant 1e-3 / 2e-3) ends with an oscillating loss: the IoU of one particular step moves by
    # up to half a point from step to step -- in the reference's own run as well (fixture trace) -- so the criterion is
    # the median over the last 200 steps; the last step's mask must lie inside the reference's own step-to-step spread.
    # It is also chaotic at the level of one fp32 rounding: three more runs of the reference itself, from parameters
    # perturbed by 1e-7, end 0.10-0.12 points away from the first (fixture "replica_traces") -- the band those runs span
    # is the reference here.
    _compare_trace(f"c3nb {precision}", trace, g["iou_trace"], g.get("replica_traces"))
    fg = _fitted_fg(m, x)
    ref_fg = synth.unpack_mask(g["mask_fg_packed"], H, W)
    iou_last = synth.fg_iou(fg, un < 0.5)
    print(f"[c3nb {precision}] last step: device {100 * iou_last:.3f}  reference {100 * g['iou_vs_unaries']:.3f}; "
          f"IoU(device mask, reference mask) {100 * synth.fg_iou(fg, ref_fg):.3f}")
    assert iou_last >= float(g["iou_trace"].min()) - 5 * MIOU_TOL
    # a non-convex target: the flow really is needed (a convex fit of this C shape stays below 0.9)
    assert float(trace.median()) > 0.97


def test_c3_flow_identity_prefit_1000_steps(A, golden):
    """``learn_flow_identity`` (1000 x Adamax 1e-2, wd 1e-5) from the reference's initial state: same ActNorm init, same first
    losses, same level at the end of the curve."""
    g = golden("full_c3nb.pt")
    H, W = g["H"], g["W"]
    m = _c3nb_model(A, g, "fp32", "init")
    x = A.GridSpecHost("index", 1, H, W).materialize(2, DEV)
    hist = m.learn_flow_identity(x, lr=1e-2, weight_decay=1e-5, max_iter=1000, use_progress_bar=False).cpu()
    ref = g["identity_hist"]
    torch.testing.assert_close(hist[0], ref[0], rtol=1e-4, atol=1e-9)
    assert float(hist[-20:].mean()) < 3.0 * float(ref[-20:].mean()) + 1e-7, (float(hist[-20:].mean()), float(ref[-20:].mean()))
    assert float(hist[-1]) < 1e-2 * float(hist[0])


@pytest.mark.parametrize("precision", ["fp32", "f16"])
def test_c2_per_frame_cold_4000_then_warm_400(A, golden, precision):
    """BASELINE configs[1]: 640x480, ConvexNextNet(L=2), Transformator grid, MSE(sigmoid(y), unaries), Adam 1e-3;
    frame 0 cold for the full 4000 steps, frame 1 warm-started from it for 400 (``path_connected_net.py:899-982``)."""
    if not os.path.exists(os.path.join(os.path.dirname(__file__), "golden", "full_c2.pt")):
        pytest.skip("full_c2.pt not generated")
    g = golden("full_c2.pt")
    H, W = g["H"], g["W"]
    sch = g["schedule"]
    m = A.ConvexNextNet(n_hidden=130, in_features=2, n_hidden_layers=2, precision=precision)
    m.load_state_dict(g["init"])
    m = m.to(DEV)
    spec = A.GridSpecHost("linspace", 1, H, W)
    fitter = None
    for k, (steps, fr) in enumerate(zip((sch["cold_steps"], sch["warm_steps"]), g["frames"])):
        un = synth.c2_unaries(H, W, seed=sch["frame_seeds"][k], t=sch["frame_t"][k])
        _check_inputs(un, fr["unaries_check"])
        if fitter is None:
            fitter = m.make_fitter(spec, un.to(DEV), A.LossConfig("mse"), A.OptimConfig("adam", lr=sch["lr"]))
        else:
            fitter.set_target(un.to(DEV))
            fitter.reset_optimizer()                      # fresh optimizer per frame (:923-933), weights carried over
        x = spec.materialize(2, DEV)
        hist, trace = _run_traced(fitter, m, x, un < 0.5, steps)
        fitter.raise_if_nonfinite()
        if k == 0:
            torch.testing.assert_close(hist[:3], fr["loss_hist"][:3], rtol=5e-3 if precision == "f16" else 1e-4, atol=1e-8)
        if "iou_trace" in fr:
            _compare_trace(f"c2 frame {k} {precision}", trace, fr["iou_trace"])
        fg = _fitted_fg(m, x)
        ref_fg = synth.unpack_mask(fr["mask_fg_packed"], H, W)
        direct = _compare(f"c2 frame {k} {precision}", fg, ref_fg, un < 0.5, fr["iou_vs_unaries"])
        assert direct > 0.99
        if precision == "f16" and k == 0:
            # The stated bound of the tensor-path logits (awb_prior_forward AWB_FWD_TC / _TC_TRAINING; include/awb.h): on
            # the weights of a finished 4000-step fit at 640x480, against the exact fp32 forward of the same weights.
            prior = m._prior_for(torch.device(DEV))
            with torch.no_grad():
                exact = m(x).reshape(-1)
                ws = prior.new_workspace(spec.n_pixels, A._lib.AWB_WS_TRAINING, torch.device(DEV))
                tp = prior.forward(m._ensure_flat(), spec, A._lib.AWB_FWD_TC, ws)[0].reshape(-1)
            per_px = float(((tp - exact).abs() / exact.abs().clamp(min=1.0)).max())
            normwise = float((tp - exact).norm() / exact.norm())
            flips = int(((tp < 0) != (exact < 0)).sum())
            print(f"[c2 tensor-path logits after 4000 steps] per-pixel |d|/max(1,|y|) max {per_px:.2e}, normwise {normwise:.2e}, "
                  f"{flips} of {exact.numel()} mask pixels differ")
            assert per_px <= TC_LOGIT_BOUND and normwise <= 1e-3 and flips <= 150      # measured 2.2e-2, 7.0e-4, 69 pixels (0.02 %)


@pytest.mark.parametrize("precision,O_", [pytest.param("fp32", 8, id="fp32"), pytest.param("f16", 8, id="f16"),
                                          pytest.param("fp32", 16, id="fp32-16objects"),
                                          pytest.param("f16", 16, id="f16-16objects")])
def test_c4_eight_grouped_realnvp_objects_equal_independent_fits(A, precision, O_):
    """BASELINE configs[3]: 8 ``real_nvp_path_connected_net`` objects of one frame fitted jointly in one grouped launch per
    kernel == 8 independent single-object fits, bit for bit (object = ``blockIdx.y``; the arithmetic per object is the
    same code path), object k against unaries channel k + 1 (``multiple_object_aware_path_connected_net.py:186-218``).
    Also with 16 objects, the most the C-ABI accepts (9 CTAs per object on the tensor path, 4 SMs idle)."""
    # tensor path: the fused kernel accumulates the weight gradients of all tiles of a CTA in TMEM, so the summation order
    # depends on how many CTAs an object gets (148 / O when grouped); it is the same -- and the fits bit-identical -- as long
    # as a frame has no more 128-pixel tiles than that share (18 for O = 8, 9 for O = 16).  Larger frames: see the next test.
    H, W = (60, 80) if precision == "fp32" else ((40, 56) if O_ == 8 else (24, 48))
    args = dict(channels=2, hidden_units=32, flow_n_flows=12, flow_output_fn="tanh", norm="minmax",
                convex_net_hidden_units=130, convex_net_hidden_layers=2, precision=precision)
    torch.manual_seed(11)
    multi = A.NumberBasedMultiPriorModule(prior_type=A.real_nvp_path_connected_net, prior_args=args, min_priors=O_).to(DEV)
    singles = []
    for k in range(O_):
        s = A.real_nvp_path_connected_net(**args)
        s.load_state_dict(multi.priors[k].state_dict())
        singles.append(s.to(DEV))
    un = synth.multi_object_unaries(H, W, O_, seed=5)[0, 1:].to(DEV)          # channel 0 is the background
    grid = A.GridSpecHost("linspace", 1, H, W)
    opt = A.OptimConfig("adamax", lr=1e-3, weight_decay=[1e-5, 0.0, 0.0, 0.0], plateau=True)
    f = multi.make_fitter(grid, un, A.LossConfig("mse"), opt, use_graph=False)      # ActNorm init of every object happens here
    hist = f.run(6)
    for k in range(O_):
        fk = singles[k].make_fitter(grid, un[k], A.LossConfig("mse"), opt, use_graph=False)
        hk = fk.run(6)
        assert torch.equal(hist[:, k], hk[:, 0]), (k, hist[:, k], hk[:, 0])
        for (name, a), b in zip(multi.priors[k].state_dict().items(), singles[k].state_dict().values()):
            assert torch.equal(a, b), f"object {k} {name}"
    x = grid.materialize(2, DEV)
    with torch.no_grad():
        out = multi(x, num_priors=O_)
        assert out.shape == (1, O_, 1, H, W)
        for k in (0, 3, O_ - 1):
            assert torch.equal(out[:, k], singles[k](x))
    # objects differ: the grouped launch did not fit one target eight times
    assert not torch.equal(hist[:, 0], hist[:, 1])


def test_c4_grouped_tensor_path_large_frame_matches_independent_fits(A):
    """Tensor path, frames with more tiles than an object's share of the SMs: grouped and independent fits differ only in
    the fp32 summation order of the weight-gradient partials -- losses agree to 1e-5 relative after 6 steps."""
    O_, H, W = 8, 96, 128
    args = dict(channels=2, hidden_units=32, flow_n_flows=12, flow_output_fn="tanh", norm="minmax",
                convex_net_hidden_units=130, convex_net_hidden_layers=2, precision="f16")
    torch.manual_seed(12)
    multi = A.NumberBasedMultiPriorModule(prior_type=A.real_nvp_path_connected_net, prior_args=args, min_priors=O_).to(DEV)
    singles = []
    for k in range(O_):
        s = A.real_nvp_path_connected_net(**args)
        s.load_state_dict(multi.priors[k].state_dict())
        singles.append(s.to(DEV))
    un = synth.multi_object_unaries(H, W, O_, seed=6)[0, 1:].to(DEV)
    grid = A.GridSpecHost("linspace", 1, H, W)
    opt = A.OptimConfig("adamax", lr=1e-3, weight_decay=[1e-5, 0.0, 0.0, 0.0], plateau=True)
    hist = multi.make_fitter(grid, un, A.LossConfig("mse"), opt, use_graph=False).run(6)
    for k in range(O_):
        hk = singles[k].make_fitter(grid, un[k], A.LossConfig("mse"), opt, use_graph=False).run(6)
        torch.testing.assert_close(hist[:, k], hk[:, 0], rtol=1e-5, atol=1e-8)
        for (name, a), b in zip(multi.priors[k].state_dict().items(), singles[k].state_dict().values()):
            torch.testing.assert_close(a, b, rtol=1e-3, atol=1e-5, msg=lambda m_: f"object {k} {name}: {m_}")
