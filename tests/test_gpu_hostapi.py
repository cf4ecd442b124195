"""GPU tests of the host-side mirror of the reference's callers: drop-in optimizers (agent loop), the per-frame /
per-sequence pretrain loops, the multi-object container with grouped launches, the device-resident prior cache."""
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


def blob(H, W, cx=0.5, cy=0.5, rx=0.27, ry=0.31, tau=0.08):
    yy, xx = torch.meshgrid(torch.linspace(0, 1, H), torch.linspace(0, 1, W), indexing="ij")
    return torch.sigmoid((torch.sqrt(((xx - cx) / rx) ** 2 + ((yy - cy) / ry) ** 2) - 1) / tau)


@pytest.mark.parametrize("kind", ["adam", "adamax"])
def test_fused_optimizer_matches_torch_in_agent_loop(A, kind):
    """optimizer_type drop-in: 3 steps of loss.backward(); optimizer.step(); enforce_convexity() on a wrapper that
    also holds a non-prior (UNet stand-in) parameter, against torch.optim on an identical copy."""
    torch.manual_seed(0)
    H, W = 40, 56
    prior = A.ConvexNextNet(n_hidden_layers=2).to(DEV)
    ref = A.ConvexNextNet(n_hidden_layers=2).to(DEV)
    ref.load_state_dict(prior.state_dict())
    extra = torch.nn.Linear(4, 4).to(DEV)
    extra_ref = torch.nn.Linear(4, 4).to(DEV)
    extra_ref.load_state_dict(extra.state_dict())
    cls = A.FusedAdam if kind == "adam" else A.FusedAdamax
    tcls = torch.optim.Adam if kind == "adam" else torch.optim.Adamax
    opt = cls([dict(params=list(prior.parameters()), weight_decay=1e-4), dict(params=list(extra.parameters()))], lr=2e-3)
    topt = tcls([dict(params=list(ref.parameters()), weight_decay=1e-4), dict(params=list(extra_ref.parameters()))], lr=2e-3)
    grid = O.grid_linspace(H, W)[None].to(DEV)
    un = blob(H, W).to(DEV)
    xin = torch.randn(8, 4, device=DEV)
    for _ in range(3):
        for m, e, o in ((prior, extra, opt), (ref, extra_ref, topt)):
            o.zero_grad()
            loss = ((torch.sigmoid(m(grid))[0, 0] - un) ** 2).mean() + e(xin).pow(2).mean()
            loss.backward()
            o.step()
            if m is ref:
                m.enforce_convexity()
    for (k, a), b in zip(prior.state_dict().items(), ref.state_dict().values()):
        torch.testing.assert_close(a, b, rtol=1e-5, atol=1e-7, msg=lambda s: f"{k}: {s}")
    for a, b in zip(extra.parameters(), extra_ref.parameters()):
        torch.testing.assert_close(a, b, rtol=1e-6, atol=1e-8)
    for k in O.icnn_clamp_keys(dict(prior.state_dict())):
        assert float(prior.state_dict()[k].min()) >= 0.0


@pytest.mark.parametrize("kind", ["adam", "adamax"])
def test_fused_optimizer_skips_a_group_without_grads_like_torch(A, kind):
    """A RealNVP prior whose flow group is frozen (grads None) on the first two steps and on step 4: torch.optim leaves
    those parameters, their moments and their step count alone, and the flow joins late and rejoins with its own count.
    A group in which only some tensors have a grad cannot be stepped as a whole: ValueError naming the tensor."""
    torch.manual_seed(0)
    H, W = 24, 32

    def make():
        torch.manual_seed(0)
        m = A.real_nvp_path_connected_net(channels=2, hidden_units=16, flow_n_flows=4, flow_output_fn="tanh",
                                          convex_net_hidden_layers=1)
        sd = m.state_dict()
        for k in sd:
            if ".net.2." in k:                                 # zero-initialised couplings would make the flow trivial
                sd[k] = 0.05 * torch.randn_like(sd[k])
            elif k.endswith("data_dep_init_done"):
                sd[k] = torch.ones_like(sd[k])
        m.load_state_dict(sd)
        return m.to(DEV)

    prior, ref = make(), make()
    cls = A.FusedAdam if kind == "adam" else A.FusedAdamax
    tcls = torch.optim.Adam if kind == "adam" else torch.optim.Adamax
    groups = lambda m: [dict(params=list(m.convex_net.parameters()), weight_decay=1e-3),
                        dict(params=list(m.flow_net.parameters()), lr=5e-3, weight_decay=1e-2),
                        dict(params=list(m.linear.parameters()))]
    opt, topt = cls(groups(prior), lr=2e-3), tcls(groups(ref), lr=2e-3)
    grid = O.grid_linspace(H, W)[None].to(DEV)
    un = blob(H, W).to(DEV)
    flow_on = [False, False, True, False, True, True]
    for on in flow_on:
        for m, o in ((prior, opt), (ref, topt)):
            m.flow_net.requires_grad_(on)
            o.zero_grad(set_to_none=True)
            ((torch.sigmoid(m(grid))[0, 0] - un) ** 2).mean().backward()
            o.step()
            if m is ref:
                m.enforce_convexity()
    for (k, a), b in zip(prior.state_dict().items(), ref.state_dict().values()):
        torch.testing.assert_close(a, b, rtol=1e-5, atol=1e-7, msg=lambda s: f"{k}: {s}")
    opt.zero_grad(set_to_none=True)
    ((torch.sigmoid(prior(grid))[0, 0] - un) ** 2).mean().backward()
    prior.convex_net.out.ln.weight.grad = None
    with pytest.raises(ValueError, match=r"convex_net\.out\.ln\.weight"):
        opt.step()


def test_fit_frames_warm_start_chain_and_skip(A):
    """_prior_based_pretrain semantics on a 4-frame synthetic sequence: cold first frame (num_epochs), warm
    successors (reuse_state_epochs), a frame without foreground is skipped and keeps the chain, IoU check passes."""
    H, W = 60, 80
    torch.manual_seed(1)
    m = A.ConvexNextNet(n_hidden_layers=2, precision="f16").to(DEV)
    frames = [blob(H, W, cx=0.45 + 0.03 * i, cy=0.5) for i in range(4)]
    frames[2] = torch.ones(H, W)                      # background only -> skipped
    grid = A.GridSpecHost("linspace", 1, H, W)
    sched = A.FitSchedule(num_epochs=600, reuse_state_epochs=150, optimizer="adam", plateau=False, lr=2e-3,
                          proper_prior_fit_threshold=0.5)
    seen = []
    res = A.fit_frames(m, [grid] * 4, frames, sched, on_frame=lambda r: seen.append(r.index))
    assert seen == [0, 1, 2, 3]
    assert [r.skipped for r in res] == [False, False, True, False]
    assert [r.steps for r in res] == [600, 150, 0, 150]
    for r in (res[0], res[1], res[3]):
        assert r.proper_fit and r.iou > 0.9, (r.index, r.iou)
        assert r.state is not None and r.state.numel() == m._arena.numel()
    # the warm fits continue from the previous frame: their first losses are far below a cold start's
    assert res[1].final_loss < 0.02 and res[3].final_loss < 0.02
    # the stored per-frame state reproduces the frame's mask
    m._arena.copy_(res[1].state)
    prob = torch.sigmoid(m(grid.materialize(2, DEV)))
    assert A.mask_iou(prob.reshape(1, -1), frames[1].to(DEV).reshape(1, -1)) == pytest.approx(res[1].iou)


def test_fit_frames_retry_after_bad_fit(A):
    """proper_prior_fit_retrys: an impossible threshold forces the reset_parameters() retry path exactly once."""
    H, W = 32, 48
    torch.manual_seed(2)
    m = A.ConvexNextNet(n_hidden_layers=1).to(DEV)
    sched = A.FitSchedule(num_epochs=20, optimizer="adam", plateau=False, proper_prior_fit_threshold=1.1,
                          proper_prior_fit_retrys=1, reuse_state=False)
    res = A.fit_frames(m, [A.GridSpecHost("linspace", 1, H, W)], [blob(H, W)], sched)
    assert res[0].retries == 1 and res[0].steps == 40 and not res[0].proper_fit


def test_fit_sequence_spatio_temporal(A):
    """_non_prior_based_pretrain: one (x,y,t) flow prior over T frames, 2 frames per step, shared optimizer state."""
    T, H, W = 6, 40, 48
    torch.manual_seed(3)
    m = A.real_nvp_path_connected_net(channels=3, hidden_units=32, flow_n_flows=6, flow_output_fn="tanh",
                                      convex_net_hidden_layers=2, precision="f16").to(DEV)
    un = torch.stack([blob(H, W, cx=0.4 + 0.04 * i) for i in range(T)])
    sched = A.FitSchedule(num_epochs=60, batch_size=2, lr=2e-3)
    hist = A.fit_sequence(m, T, H, W, un, sched)
    assert hist.numel() == 60 * 3 and bool(torch.isfinite(hist).all())
    assert float(hist[-3:].mean()) < 0.5 * float(hist[:3].mean())
    # t really enters: the fitted masks follow the moving blob
    grid = A.GridSpecHost("linspace", T, H, W, t0=0.0, t_step=1.0 / (T - 1)).materialize(3, DEV)
    prob = torch.sigmoid(m(grid))[:, 0]
    cx = [float((1 - p).mul(torch.linspace(0, 1, W, device=DEV)).sum() / (1 - p).sum()) for p in prob]
    assert cx[-1] > cx[0] + 0.05, cx


@pytest.mark.parametrize("precision", ["fp32", "f16"])
def test_multi_object_grouped_fit_equals_independent_fits(A, precision):
    """Config 4 semantics: O priors fitted jointly in one grouped launch == O independent single-object fits
    (bit for bit: the object index is a grid dimension, the arithmetic per object is unchanged)."""
    O_, H, W = 3, 48, 64
    torch.manual_seed(4)
    multi = A.NumberBasedMultiPriorModule(prior_type=A.ConvexNextNet,
                                          prior_args=dict(n_hidden_layers=2, precision=precision), min_priors=O_).to(DEV)
    singles = []
    for k in range(O_):
        s = A.ConvexNextNet(n_hidden_layers=2, precision=precision).to(DEV)
        s.load_state_dict(multi.priors[k].state_dict())
        singles.append(s)
    un = torch.stack([blob(H, W, cx=0.3 + 0.2 * k, rx=0.15, ry=0.2) for k in range(O_)]).to(DEV)
    grid = A.GridSpecHost("linspace", 1, H, W)
    f = multi.make_fitter(grid, un, A.LossConfig("mse"), A.OptimConfig("adam", lr=1e-3), use_graph=False)
    hist = f.run(5)
    for k in range(O_):
        fk = singles[k].make_fitter(grid, un[k], A.LossConfig("mse"), A.OptimConfig("adam", lr=1e-3), use_graph=False)
        hk = fk.run(5)
        assert torch.equal(hist[:, k], hk[:, 0]), (k, hist[:, k], hk[:, 0])
        for (name, a), b in zip(multi.priors[k].state_dict().items(), singles[k].state_dict().values()):
            assert torch.equal(a, b), f"object {k} {name}"
    out = multi(grid.materialize(2, DEV), num_priors=O_)
    assert out.shape == (1, O_, 1, H, W)
    torch.testing.assert_close(out[:, 1], singles[1](grid.materialize(2, DEV)))
    assert list(multi.state_dict().keys())[0] == "priors.0.input.weight"


def test_device_prior_cache_and_manager(A):
    """Per-frame weight swap as row copies; on-disk format of the reference's PriorCache."""
    import io
    torch.manual_seed(5)
    m = A.ConvexNextNet(n_hidden_layers=2).to(DEV)
    cache = A.DevicePriorCache(A.ConvexNextNet, dict(n_hidden_layers=2), capacity=2)
    H, W = 24, 32
    grid = A.GridSpecHost("linspace", 1, H, W)
    states = {}
    for key in (7, 3, 11):                # more frames than the initial capacity
        with A.PriorManager(m, prior_state=(key, None), prior_cache=cache, training=True):
            f = m.make_fitter(grid, blob(H, W, cx=0.3 + 0.02 * key).to(DEV), A.LossConfig("mse"), A.OptimConfig("adam"),
                              use_graph=False)
            f.run(3)
            states[key] = {k: v.detach().clone() for k, v in m.state_dict().items()}
    for key in (3, 7, 11):
        with A.PriorManager(m, prior_state=(key, None), prior_cache=cache):
            for k, v in m.state_dict().items():
                assert torch.equal(v, states[key][k]), (key, k)
    buf = io.BytesIO()
    cache.save(buf)
    buf.seek(0)
    st = torch.load(buf, map_location="cpu", weights_only=False)
    assert set(st) == {"model_type", "model_args", "store_device", "cache"} and set(st["cache"]) == {"7", "3", "11"}
    assert st["model_type"].endswith("ConvexNextNet")
    for k, v in states[11].items():
        assert torch.equal(st["cache"]["11"][k], v.cpu())


def test_joint_trainer_matches_manual_agent_step(A):
    """Config 5 on one rank: JointTrainer(FusedAdam, grads as bucket views) == the reference's step written out by hand
    (zero_grad; cat(sigmoid(seg), sigmoid(prior)); FBMSJointLoss; backward; Adam.step; enforce_convexity)."""
    from awesome_b200 import measures as M
    torch.manual_seed(6)
    B, H, W = 2, 32, 40

    def nets():
        torch.manual_seed(6)
        seg = torch.nn.Sequential(torch.nn.Conv2d(4, 8, 3, padding=1), torch.nn.ReLU(), torch.nn.Conv2d(8, 1, 3, padding=1)).to(DEV)
        pri = A.real_nvp_path_connected_net(channels=3, hidden_units=32, flow_n_flows=6, flow_output_fn="tanh",
                                            convex_net_hidden_layers=2).to(DEV)
        return seg, pri

    g = torch.Generator().manual_seed(0)
    img = torch.randn(B, 4, H, W, generator=g).to(DEV)
    grid = A.GridSpecHost("linspace", B, H, W, t0=0.2, t_step=0.1).materialize(3, DEV)
    lab = torch.full((B, 1, H, W), 2.0)
    lab[torch.rand(B, 1, H, W, generator=g) < 0.15] = 0.0
    lab[torch.rand(B, 1, H, W, generator=g) < 0.3] = 1.0
    lab = lab.to(DEV)

    seg, pri = nets()
    pri(grid)                                            # ActNorm data-dependent init happens on the first forward
    tr = A.JointTrainer(seg, pri, M.FBMSJointLoss(), optimizer_args=dict(lr=1e-3))
    l_ours = [float(tr.step(img, grid, lab)) for _ in range(3)]

    seg2, pri2 = nets()
    pri2(grid)
    opt = torch.optim.Adam(list(seg2.parameters()) + list(pri2.parameters()), lr=1e-3)
    crit = M.FBMSJointLoss()
    l_ref = []
    for _ in range(3):
        opt.zero_grad()
        out = torch.cat([torch.sigmoid(seg2(img)), torch.sigmoid(pri2(grid))], 1)
        loss = crit(out, lab)
        loss.backward()
        opt.step()
        pri2.enforce_convexity()
        l_ref.append(float(loss))
    torch.testing.assert_close(torch.tensor(l_ours), torch.tensor(l_ref), rtol=1e-5, atol=1e-7)
    for (k, a), b in zip(pri.state_dict().items(), pri2.state_dict().values()):
        if a.dtype.is_floating_point:
            torch.testing.assert_close(a, b, rtol=1e-4, atol=2e-6, msg=lambda s: f"{k}: {s}")
    for a, b in zip(seg.parameters(), seg2.parameters()):
        torch.testing.assert_close(a, b, rtol=1e-5, atol=1e-7)
    assert tr.bucket.nbytes == 4 * sum(p.numel() for p in list(seg.parameters()) + list(pri.parameters()))


class _FakeWrapper(torch.nn.Module):
    """Stands in for the reference WrapperModule on the pretrain path: with evaluate_prior=False the call returns the
    segmentation unaries [B,1,H,W] (wrapper_module.py:157-228); get_prior_args hands out the coordinate grid."""

    def __init__(self):
        super().__init__()
        self.evaluate_prior = True
        self.dummy = torch.nn.Parameter(torch.zeros(1))

    def forward(self, image, grid):
        assert self.evaluate_prior is False
        return image[:, :1]                       # the "UNet" output is stored in the image's first channel

    def get_prior_args(self, image, grid, segm=None):
        return (grid,), {}


class _FakeDataset(torch.utils.data.Dataset):
    def __init__(self, frames, grid, cache):
        self.frames, self.grid = frames, grid
        self.__prior_cache__ = cache
        self.has_prior = cache is not None

    def __len__(self):
        return len(self.frames)

    def __getitem__(self, i):
        return (i, 0), ((self.frames[i][None], self.grid[0]), torch.zeros(1))


class _FakeAgent:
    def __init__(self, ds):
        self.training_dataset = ds

    def _decompose_training_item(self, item):
        (key, _state), (inputs, labels) = item
        return list(inputs), labels, None, (int(key), None)


@pytest.mark.parametrize("kind", ["pcn", "diffeo"])
def test_pretrain_protocol_with_duck_typed_agent(A, kind):
    """PretrainableModule.pretrain(train_set, test_set, device, agent, use_progress_bar, wrapper_module=..., **args):
    per-frame states land in the dataset's prior cache and come back in the reference's PriorCache state format."""
    H, W = 40, 56
    torch.manual_seed(7)
    if kind == "pcn":
        m = A.real_nvp_path_connected_net(channels=2, hidden_units=32, flow_n_flows=6, flow_output_fn="tanh",
                                          convex_net_hidden_layers=2, precision="f16").to(DEV)
        typ, args = A.real_nvp_path_connected_net, dict(channels=2, hidden_units=32, flow_n_flows=6, flow_output_fn="tanh")
    else:
        m = A.ConvexDiffeomorphismNet(n_hidden_layers=1, precision="f16").to(DEV)
        typ, args = A.ConvexDiffeomorphismNet, dict(n_hidden_layers=1)
    frames = [blob(H, W, cx=0.45 + 0.05 * i) for i in range(3)]
    grid = A.GridSpecHost("linspace", 1, H, W).materialize(2, "cpu")
    cache = A.DevicePriorCache(typ, args)
    ds = _FakeDataset(frames, grid, cache)
    state = m.pretrain(ds, None, torch.device(DEV), _FakeAgent(ds), use_progress_bar=False, wrapper_module=_FakeWrapper().to(DEV),
                       num_epochs=300, reuse_state_epochs=80, lr=3e-3, proper_prior_fit_threshold=0.5,
                       prefit_flow_net_identity=(kind == "pcn"), prefit_flow_net_identity_num_epochs=20,
                       prefit_convex_net=(kind == "pcn"), prefit_convex_net_num_epochs=30)
    assert set(state) == {"model_type", "model_args", "store_device", "cache"} and set(state["cache"]) == {"0", "1", "2"}
    # every stored frame state reproduces that frame's mask
    for i in range(3):
        m.load_state_dict(state["cache"][str(i)])
        prob = torch.sigmoid(m(grid.to(DEV)))
        assert A.mask_iou(prob.reshape(1, -1), frames[i].to(DEV).reshape(1, -1)) > 0.85, (kind, i)
    # and pretrain_load_state puts them back into a fresh cache
    cache2 = A.DevicePriorCache(typ, args)
    ds2 = _FakeDataset(frames, grid, cache2)
    m.pretrain_load_state(ds2, None, torch.device(DEV), _FakeAgent(ds2), state, wrapper_module=None)
    assert 1 in cache2 and torch.equal(cache2[1]["convex_net.input.weight"].cpu(), state["cache"]["1"]["convex_net.input.weight"])


@pytest.mark.parametrize("precision", ["fp32", "f16"])
def test_host_frame_fit_equals_device_frame_fit(A, precision):
    """awb_prior_fit_host_frames (host unaries, copy stream + double-buffered staging, losses stored into pinned host
    memory) == the same frames fitted one step at a time from device memory, bit for bit: parameters and losses."""
    torch.manual_seed(3)
    H, W = 48, 72
    frames = [blob(H, W, cx=0.4 + 0.05 * k, ry=0.25 + 0.02 * k).reshape(1, -1).contiguous() for k in range(3)]
    pinned = [f.pin_memory() if k != 1 else f for k, f in enumerate(frames)]      # one pageable frame: still correct
    grid = A.GridSpecHost("linspace", 1, H, W)
    steps = 7
    m1 = A.ConvexNextNet(n_hidden_layers=2, precision=precision).to(DEV)
    m2 = A.ConvexNextNet(n_hidden_layers=2, precision=precision).to(DEV)
    m2.load_state_dict(m1.state_dict())
    f1 = m1.make_fitter(grid, frames[0].to(DEV), A.LossConfig("mse"), A.OptimConfig("adam", lr=1e-3), use_graph=False)
    f2 = m2.make_fitter(grid, frames[0].to(DEV), A.LossConfig("mse"), A.OptimConfig("adam", lr=1e-3), use_graph=False)
    ref_losses = []
    for s in range(steps):
        f1.set_target(frames[s % 3].to(DEV))
        ref_losses.append(f1.run(1)[0].cpu())
    got = f2.run_host_frames(pinned, steps)
    torch.cuda.synchronize()
    assert got.shape == (steps, 1) and got.is_pinned()
    torch.testing.assert_close(got, torch.stack(ref_losses), rtol=0, atol=0)
    for (k, a), b in zip(m1.state_dict().items(), m2.state_dict().values()):
        assert torch.equal(a, b), k
    assert f2.steps_done == steps
    from awesome_b200 import _lib as AL
    import ctypes as C
    with pytest.raises(AL.AwbError):     # the loss slots must be device-mapped host memory
        lib = f2.lib
        ptrs = (C.c_void_p * 1)(pinned[0].data_ptr())
        bad = torch.empty(4)
        AL.check(lib.awb_prior_fit_host_frames(f2.prior.handle, f2.params.data_ptr(), f2.opt_state.data_ptr(),
                                                   C.byref(f2._gs), ptrs, 1, 1, f2._specs, C.byref(f2._hyper),
                                                   bad.data_ptr(), f2._staging.data_ptr(), f2.ws.data_ptr(),
                                                   f2.ws.numel(), 0, AL.stream_ptr()))


def test_grouped_frames_one_wave_at_frame_size_matches_single_frame_fits(A):
    """Four independent 640x480 frames per fused launch run as ONE wave (37 persistent CTAs per frame instead of 148): the
    gradient partials are summed in a different grouping than in a one-frame launch, so parity with four separate
    fits is to fp32 summation order -- losses to 1e-5 relative, parameters to 2e-5 after 6 Adam steps (lr 1e-3 moves a
    weight by <= 6e-3, so this is a tight bound on the gradients' sign and size), logits to 1e-3 -- and repeatable bit for bit."""
    G, H, W = 4, 480, 640
    torch.manual_seed(11)
    multi = A.NumberBasedMultiPriorModule(prior_type=A.ConvexNextNet,
                                          prior_args=dict(n_hidden_layers=2, precision="f16"), min_priors=G).to(DEV)
    start = [{k: v.clone() for k, v in p.state_dict().items()} for p in multi.priors]
    un = torch.stack([blob(H, W, cx=0.35 + 0.08 * k, cy=0.45 + 0.03 * k, rx=0.2, ry=0.26) for k in range(G)]).to(DEV)
    grid = A.GridSpecHost("linspace", 1, H, W)
    f = multi.make_fitter(grid, un, A.LossConfig("mse"), A.OptimConfig("adam", lr=1e-3), use_graph=False)
    hist = f.run(6).clone()
    grouped = [{k: v.clone() for k, v in p.state_dict().items()} for p in multi.priors]
    for k in range(G):
        s = A.ConvexNextNet(n_hidden_layers=2, precision="f16").to(DEV)
        s.load_state_dict(start[k])
        hk = s.make_fitter(grid, un[k], A.LossConfig("mse"), A.OptimConfig("adam", lr=1e-3), use_graph=False).run(6)
        torch.testing.assert_close(hist[:, k], hk[:, 0], rtol=1e-5, atol=1e-8)
        for name, b in s.state_dict().items():
            torch.testing.assert_close(grouped[k][name], b, rtol=0, atol=2e-5, msg=lambda m: f"frame {k} {name}: {m}")
    # determinism of the grouped launch itself
    for p, st in zip(multi.priors, start):
        p.load_state_dict(st)
    f2 = multi.make_fitter(grid, un, A.LossConfig("mse"), A.OptimConfig("adam", lr=1e-3), use_graph=False)
    assert torch.equal(f2.run(6), hist)
    for p, st in zip(multi.priors, grouped):
        for name, b in p.state_dict().items():
            assert torch.equal(st[name], b), name


def test_no_grad_forward_is_exact_fp32_on_cached_workspace(A):
    """A forward under ``torch.no_grad()`` of a module whose parameters require grad takes the inference path: exact fp32
    logits (also for precision="f16") on the cached workspace, no training-sized allocation (ADVICE r1)."""
    torch.manual_seed(0)
    m32 = A.ConvexNextNet(n_hidden_layers=2).to(DEV)
    m16 = A.ConvexNextNet(n_hidden_layers=2, precision="f16")
    m16.load_state_dict(m32.state_dict())
    m16 = m16.to(DEV)
    x = A.GridSpecHost("linspace", 1, 40, 56).materialize(2, DEV)
    with torch.no_grad():
        y32, y16 = m32(x), m16(x)
        ws = m16._prior._ws_cache
        assert len(ws) == 1 and list(ws.keys())[0][1] == A._lib.AWB_WS_INFERENCE   # inference workspace, cached
        y16b = m16(x)
        assert len(m16._prior._ws_cache) == 1
    assert torch.equal(y32, y16) and torch.equal(y16, y16b)               # bit-identical: same fp32 kernels
    assert not y16.requires_grad
    y_train = m16(x)                                                     # grad enabled: tensor-path logits, differentiable
    assert y_train.requires_grad
    assert float((y_train - y32).abs().max()) < 2e-2
    # a workspace layout or forward mode outside the named ones is refused, not mapped to a neighbouring one
    L, prior = A._lib, m16._prior
    for layout in (L.AWB_WS_INFERENCE - 1, L.AWB_WS_SECOND_ORDER + 1):
        assert prior.lib.awb_prior_workspace_bytes(prior.handle, 40 * 56, layout) == -1
    ws = prior.new_workspace(40 * 56, L.AWB_WS_SECOND_ORDER, DEV)
    with pytest.raises(L.AwbError, match="unknown forward mode 4") as err:
        prior.forward(m16._ensure_flat(), A.GridSpecHost("linspace", 1, 40, 56), L.AWB_FWD_TC_TRAINING + 1, ws)
    assert err.value.code == -1                                          # AWB_ERR_INVALID


def test_pixel_row_input_gradient_shape_and_values(A):
    """``forward([N,C])`` with ``requires_grad`` rows: the input gradient comes back as ``[N,C]`` and equals the
    ``[B,C,H,W]`` path's (``model_input_requires_grad`` configs; ADVICE r1)."""
    torch.manual_seed(1)
    m = A.ConvexNextNet(n_hidden_layers=2).to(DEV)
    H, W = 12, 20
    x4 = A.GridSpecHost("linspace", 1, H, W).materialize(2, DEV).clone().requires_grad_(True)
    rows = x4.detach().permute(0, 2, 3, 1).reshape(-1, 2).clone().requires_grad_(True)
    wgt = torch.linspace(-1, 1, H * W, device=DEV)
    (m(x4).reshape(-1) * wgt).sum().backward()
    y = m(rows)
    assert y.shape == (H * W, 1)
    (y.reshape(-1) * wgt).sum().backward()
    assert rows.grad.shape == rows.shape
    torch.testing.assert_close(rows.grad, x4.grad.permute(0, 2, 3, 1).reshape(-1, 2), rtol=1e-5, atol=1e-7)
    p = O.clone_params({k: v.detach().cpu() for k, v in m.state_dict().items()})
    r = rows.detach().cpu().clone().requires_grad_(True)
    (O.icnn_forward(p, r).reshape(-1) * wgt.cpu()).sum().backward()
    torch.testing.assert_close(rows.grad.cpu(), r.grad, rtol=1e-4, atol=1e-6)


@pytest.mark.parametrize("cls_name", ["FusedAdam", "FusedAdamax"])
def test_fused_optimizer_state_dict_round_trip(A, cls_name):
    """save -> recreate -> load_state_dict -> the next step is bit-equal to the uninterrupted run, for the arena parameters
    (native moments blob) and for ordinary parameters (stock inner optimizer) -- what the agent does around every
    best-model save (torch_agent.py:356, 808, 836; ADVICE r1)."""
    cls = getattr(A, cls_name)
    x = A.GridSpecHost("linspace", 1, 24, 32).materialize(2, DEV)
    tgt = blob(24, 32).to(DEV)[None, None]

    def make():
        torch.manual_seed(5)
        prior = A.ConvexNextNet(n_hidden_layers=2).to(DEV)
        other = torch.nn.Linear(3, 2).to(DEV)
        opt = cls([dict(params=list(other.parameters())), dict(params=list(prior.parameters()))], lr=2e-3)
        return prior, other, opt

    def one_step(prior, other, opt):
        opt.zero_grad()
        loss = ((torch.sigmoid(prior(x)) - tgt) ** 2).mean() + other(torch.ones(1, 3, device=DEV)).pow(2).sum()
        loss.backward()
        opt.step()
        prior.enforce_convexity()

    pa, oa, opta = make()
    for _ in range(3):
        one_step(pa, oa, opta)
    sd = opta.state_dict()
    assert sd["awb_fused"]["native"][0]["blob"] is not None and sd["awb_fused"]["inner"] is not None
    weights = ({k: v.clone() for k, v in pa.state_dict().items()}, {k: v.clone() for k, v in oa.state_dict().items()})
    one_step(pa, oa, opta)                                   # uninterrupted 4th step
    pb, ob, optb = make()                                    # fresh objects, as after _free_optimizer / _get_optimizer
    pb.load_state_dict(weights[0]); ob.load_state_dict(weights[1])
    optb.load_state_dict(sd)
    one_step(pb, ob, optb)
    for (k, a), b in zip(pa.state_dict().items(), pb.state_dict().values()):
        assert torch.equal(a, b), k
    for (k, a), b in zip(oa.state_dict().items(), ob.state_dict().values()):
        assert torch.equal(a, b), k
    # without the saved moments the step differs (the test would be vacuous otherwise)
    pc, oc, optc = make()
    pc.load_state_dict(weights[0]); oc.load_state_dict(weights[1])
    one_step(pc, oc, optc)
    assert not torch.equal(pa.state_dict()["input.weight"], pc.state_dict()["input.weight"])
