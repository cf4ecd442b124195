"""Launch regimes of the fit-path kernels against a float64 reference.

Every fit-path kernel picks its launch geometry, and sometimes its code path, from the problem size on the host
(``awb_flow.cu``, ``awb_tc_fit.cu``, ``awb_internal.cuh``).  Each case below is a shape on ONE side of such a branch:
the shared-memory / global-memory variants of the RealNVP backward (``k_flow_bwd<3>``, ``k_flow_bwd<2>``,
``k_flow_bwd_seg``), empty and ragged pixel ranges, full / remainder rounds, and the tile and CTA edges of the tensor path.
``regime()`` restates the host formulas; every case names the branch it is meant to hit and the test asserts that the
restatement agrees, so a case fails loudly if the constants move instead of quietly covering something else.

The reference is ``oracle/prior_oracle.py`` run in float64 on the GPU with plain torch autograd.  The exact fp32 path is
compared per entry (``|g - g64| <= tol * max|g64|`` per tensor) with one set of tolerances for every regime, calibrated on
the 640x480 C = 2 frame that the rest of the suite already covers.  A float64-only self-check proves that the gradient
tolerance can see one dropped (or doubled) pixel range of the backward.  The tensor path (fp16 operands) is compared on its
loss, and on its gradients at the normwise bounds of DESIGN section 4.  Generated grids are checked bit for bit against the
same grid built by torch and passed explicitly, also through ``slice_grads`` windows that start mid-frame and mid-row."""
import pytest
import torch

import __graft_entry__ as entry
from oracle import prior_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# Exact fp32 path against float64, per entry relative to the largest reference entry of the tensor.  Calibrated on the
# regime the rest of the suite already covers (C = 2 flow prior, 1 x 480 x 640, case ``calib``), measured on one B200:
# gradients 3.4e-5, logits / deformation 9.7e-7, loss 5.7e-8; the bounds below leave a margin of 15x to 20x.  One set for
# every regime: a branch-specific bug shows up as an outlier.  (Dropping the backward's last pixel range moves some gradient
# entry by 8e-3 or more in every case: the self-check below.)
TOL_GRAD = 5e-4          # parameter gradients (autograd backward and fused step)
TOL_FWD = 2e-5           # logits and flow deformation
TOL_LOSS = 1e-6          # loss of the fused step, relative
# Tensor path (fp16 operands, fp32 accumulation): loss relative to float64 (measured <= 4.5e-5; one dropped tile of 148 moves
# it by ~7e-3); gradients at the normwise bounds of DESIGN section 4 -- per tensor for the ICNN, over the flow's parameters
# as one block and per tensor with a floor (a flow bias whose pixel sum cancels can be off by several percent of its own
# small norm at fp16 precision).
TC_TOL_LOSS = 2e-4
TC_TOL_GRAD_ICNN, TC_TOL_GRAD_FLOW = 1e-2, 2e-2
# Each flow tensor is also held to TC_TOL_GRAD_FLOW on its own, relative to max(its norm, TC_FLOW_FLOOR x the block's norm):
# an error confined to one small tensor (ActNorm, linear) must stay below 2e-3 of the block, ten times less than the block
# check alone would let through.
TC_FLOW_FLOOR = 0.1
TC_LOGIT_BOUND = 3e-2    # per pixel |d| / max(1, |y|), include/awb.h


@pytest.fixture(scope="module", autouse=True)
def built():
    entry.build()


@pytest.fixture(scope="module")
def A():
    import awesome_b200
    return awesome_b200


# ----------------------------------------------------------------------------------------------- host dispatch, restated
K_MAX_SPLITS = 148            # awb_internal.cuh kMaxSplits
FLOW_P = FLOW_PB = 4          # awb_flow.cu: pixels per thread and full round, forward / backward
FLOW_BWD_T = 256              # awb_flow.cu FLOW_BWD_T
FLOW_RED_FLOATS = 16 * 128 + 16 * 16
FLOW_TAB, FLOW_SEG_ROWS, FLOW_SEG_RS = 456, 132, 144
DZ_SMEM_LIMIT = 200 * 1024    # flow_bwd_dz_in_smem
SEG_SMEM_LIMIT = 220 * 1024   # flow_backward's limit for flow_seg_bwd_smem


def cdiv(a, b):
    return (a + b - 1) // b


def round_up(a, b):
    return cdiv(a, b) * b


def n_splits(n):
    """awb_internal.cuh ``n_splits``: pixel ranges of the cross-pixel reductions."""
    return max(1, min(cdiv(n, 256), K_MAX_SPLITS))


def split_chunk(n):
    """awb_internal.cuh ``split_chunk``: rows per range, rounded up to 8 (trailing ranges can be empty)."""
    return round_up(cdiv(n, n_splits(n)), 8)


def flow_bwd_smem_base(C, F):
    """awb_flow.cu ``flow_bwd_smem_base``: k_flow_bwd's shared memory without the running gradient."""
    stride = 32 * (8 if C == 2 else 12) + 4                       # FlowBwdPack<C>::flow_stride
    rw = 4 if C == 2 else 8                                        # FlowSave<C>::RW
    return 4 * (F * stride + 2 * FLOW_RED_FLOATS + 2 * FLOW_PB * rw * FLOW_BWD_T)


def flow_bwd_dz_in_smem(C, F, n):
    """awb_flow.cu ``flow_bwd_dz_in_smem``: the running gradient (and C = 3's pass partial) of a range fits on the SM."""
    return flow_bwd_smem_base(C, F) + 4 * split_chunk(n) * C * (2 if C == 3 else 1) <= DZ_SMEM_LIMIT


def flow_seg_bwd_smem(F, chunk_in_smem, T=FLOW_BWD_T):
    """awb_flow.cu ``flow_seg_bwd_smem``: k_flow_bwd_seg's shared memory, held against 220 KiB."""
    return 4 * (F * (FLOW_TAB + 4) + 64 + 2 * FLOW_PB * T * 4 + max(FLOW_SEG_ROWS * T, F * FLOW_SEG_RS) + 2 * chunk_in_smem)


def flow_tables(C, precision, flow_eval):
    """awb_flow.cu ``flow_seg_path`` / ``flow_seg3_path`` (m = 32, tanh couplings, output scale 1)."""
    return flow_eval == 2 or (flow_eval == 0 and precision == "f16")


def flow_fwd_geometry(n, O, tables, sms):
    """awb_flow.cu ``flow_forward``: k CTAs per SM (1..8), chunk >= 32, T, R full rounds of FLOW_P, rounds1 remainder."""
    T = 256 if tables else 128
    per_sm = cdiv(n * O, sms)
    k = min(max((per_sm + FLOW_P * T // 2) // (FLOW_P * T), 1), 8)
    n_cta = max(sms * k // O, 1)
    chunk = max(cdiv(n, n_cta), 32)
    S = cdiv(n, chunk)
    if chunk < T:
        T = round_up(chunk, 32)
    R = chunk // (FLOW_P * T)
    return dict(k=k, chunk=chunk, S=S, T=T, R=R, rounds1=cdiv(chunk - R * FLOW_P * T, T))


def flow_bwd_geometry(C, F, n, seg):
    """awb_flow.cu ``flow_backward``: which kernel variant, and its ranges / rounds."""
    S, chunk = n_splits(n), split_chunk(n)
    if seg:
        T = FLOW_BWD_T
        wl = cdiv(chunk, FLOW_BWD_T // 32)
        R = wl // (32 * FLOW_PB)
        rounds1 = cdiv(wl - R * 32 * FLOW_PB, 32)
        dz_smem = flow_seg_bwd_smem(F, chunk) <= SEG_SMEM_LIMIT
        kernel = f"k_flow_bwd_seg<{'true' if dz_smem else 'false'}>"
    else:
        T = round_up(chunk, 32) if chunk < FLOW_BWD_T else FLOW_BWD_T
        R = chunk // (FLOW_PB * T)
        rounds1 = cdiv(chunk - R * FLOW_PB * T, T)
        dz_smem = flow_bwd_dz_in_smem(C, F, n)
        kernel = f"k_flow_bwd<{C}>"
    nonempty = cdiv(n, chunk)
    return dict(kernel=kernel, dz_smem=dz_smem, S=S, chunk=chunk, T=T, R=R, rounds1=rounds1, empty=S - nonempty,
                last=((nonempty - 1) * chunk, n))


def tc_geometry(n, O, sms):
    """awb_tc_fit.cu ``tc_fit_forward_backward``: 128-row tiles, min(n_tiles, sms / O) persistent CTAs per object."""
    n_tiles = cdiv(n, 128)
    return dict(n_tiles=n_tiles, grid=min(n_tiles, max(sms // O, 1)), rem=n % 128)


def regime(case, sms):
    """Flat dict of everything the host decides for this case (keys ``fwd.*``, ``bwd.*``, ``tc.*``)."""
    n = case["B"] * case["H"] * case["W"]
    out = {"N": n}
    if case["kind"] == "flow":
        tables = flow_tables(case["C"], case["precision"], case.get("flow_eval", 0))
        out.update({f"fwd.{k}": v for k, v in flow_fwd_geometry(n, case.get("O", 1), tables, sms).items()})
        seg = tables and case["C"] == 2            # C = 3 keeps the unit loops in the backward
        out.update({f"bwd.{k}": v for k, v in flow_bwd_geometry(case["C"], case["F"], n, seg).items()})
    else:
        out.update({f"bwd.{k}": v for k, v in flow_bwd_geometry(2, 0, n, False).items() if k in ("S", "chunk", "empty", "last")})
    if case["precision"] == "f16":
        out.update({f"tc.{k}": v for k, v in tc_geometry(n, case.get("O", 1), sms).items()})
    return out


def check_regime(case):
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    r = regime(case, sms)
    for key, want in case["expect"].items():
        assert r[key] == want, f"{case['id']}: meant to cover {case['branch']}, but {key} = {r[key]} (expected {want})"
    return r


# ------------------------------------------------------------------------------------------------------- priors, inputs
def make_models(A, case, seed=0):
    """``O`` priors of the case's configuration with non-trivial couplings and ActNorm, in state_dict order."""
    models = []
    for o in range(case.get("O", 1)):
        torch.manual_seed(seed + 17 * o)
        if case["kind"] == "flow":
            m = A.real_nvp_path_connected_net(channels=case["C"], hidden_units=32, flow_n_flows=case["F"], flow_output_fn="tanh",
                                              norm="minmax", convex_net_hidden_units=130, convex_net_hidden_layers=case["L"],
                                              precision=case["precision"])
            sd = m.state_dict()
            for k in sd:
                if ".net.2." in k:                                 # zero-initialised couplings would make the flow trivial
                    sd[k] = 0.05 * torch.randn_like(sd[k])
                elif k.endswith((".s", ".t")) and ".flows." in k:  # ActNorm
                    sd[k] = 0.1 * torch.randn_like(sd[k])
                elif k.endswith("data_dep_init_done"):
                    sd[k] = torch.ones_like(sd[k])
            m.load_state_dict(sd)
        else:
            m = A.ConvexNextNet(in_features=case["C"], n_hidden_layers=case["L"], precision=case["precision"])
        models.append(m.to(DEV))
    return models


def make_handle(A, case, models):
    """One native handle for the ``O`` objects (grouped launch) and the ``[O, P]`` parameter arena."""
    L = A._lib
    prec = L.AWB_PREC_F16 if case["precision"] == "f16" else L.AWB_PREC_FP32
    if case["kind"] == "flow":
        prior = A.Prior(L.AWB_KIND_FLOW_ICNN, case["C"], 130, case["L"], n_flows=case["F"], flow_hidden=32, flow_tanh=True,
                        n_objects=len(models), precision=prec)
        models[0].flow_eval = case.get("flow_eval", 0)
        models[0]._push_consts(prior)
    else:
        prior = A.Prior(L.AWB_KIND_ICNN, case["C"], 130, case["L"], n_objects=len(models), precision=prec)
    params = torch.stack([m._ensure_flat().detach() for m in models]).contiguous()
    assert params.shape[1] == prior.n_params
    return prior, params


T0, T_STEP = 0.1, 0.3        # t channel of C = 3 grids (t_step != 0; b * t_step is exact for b <= 2)


def grid_spec(A, case, mode="linspace"):
    return A.GridSpecHost(mode, case["B"], case["H"], case["W"], t0=T0, t_step=T_STEP)


def torch_grid(mode, B, H, W, C_, t0=T0, t_step=T_STEP):
    """``[B, C, H, W]`` fp32: what a generated grid stands for, built by torch (x = linspace / index over W, y over H,
    t = t0 + b * t_step in fp32)."""
    if mode == "linspace":
        y, x = torch.linspace(0, 1, H), torch.linspace(0, 1, W)
    else:
        y, x = torch.arange(H).float() / H, torch.arange(W).float() / W
    yy, xx = torch.meshgrid(y, x, indexing="ij")
    ch = [xx.expand(B, H, W), yy.expand(B, H, W)]
    if C_ == 3:
        t = torch.full((B,), t0, dtype=torch.float32) + torch.arange(B, dtype=torch.float32) * torch.tensor(t_step)
        ch.append(t.view(B, 1, 1).expand(B, H, W))
    return torch.stack(ch, 1).contiguous().to(DEV)


def make_target(case):
    B, H, W = case["B"], case["H"], case["W"]
    yy, xx = torch.meshgrid(torch.linspace(0, 1, H), torch.linspace(0, 1, W), indexing="ij")
    out = []
    for o in range(case.get("O", 1)):
        fr = [torch.sigmoid((torch.sqrt(((xx - 0.4 - 0.05 * b - 0.02 * o) / 0.22) ** 2 + ((yy - 0.5) / 0.27) ** 2) - 1) / 0.08)
              for b in range(B)]
        out.append(torch.stack(fr).reshape(-1))
    return torch.stack(out).contiguous().to(DEV)


# ---------------------------------------------------------------------------------------------------- float64 reference
def reference(model, kind, rows, target, last, chunk_rows=1 << 18):
    """float64 oracle of one object on pixel rows ``[N, C]``: logits, deformation, loss (SE of the sigmoid, mean), every
    parameter gradient, and the gradient with the rows ``last = (r0, r1)`` removed from the loss (same 1/N).  Rows are
    processed in chunks (one of them exactly ``last``); the gradients of the chunks are added in float64."""
    names = [k for k, _ in model.named_parameters()]
    p = {k: v.detach().to(DEV, torch.float64).clone() for k, v in model.state_dict().items()}
    for k in names:
        p[k].requires_grad_(True)
    N, C_ = rows.shape
    r0, r1 = last
    bounds = sorted({0, N, r0, r1} | set(range(0, r0, chunk_rows)) | set(range(r0, r1, chunk_rows)))
    grads = [torch.zeros_like(p[k]) for k in names]
    g_last = [torch.zeros_like(p[k]) for k in names]
    logits, deformed, loss = [], [], 0.0
    for a, b in zip(bounds[:-1], bounds[1:]):
        x = rows[a:b].double().t().reshape(1, C_, 1, b - a)       # pixel rows as a [1, C, 1, n] grid, like the module does
        if kind == "flow":
            xd = O.pathconnected_deformation(p, x)
            y = O.icnn_forward(p, xd, "convex_net.").reshape(-1)
            deformed.append(xd.detach())
        else:
            y = O.icnn_forward(p, O.pixelize(x)).reshape(-1)
        l = ((target[a:b].double() - torch.sigmoid(y)) ** 2).sum() / N
        gs = torch.autograd.grad(l, [p[k] for k in names])
        for acc, g in zip(grads, gs):
            acc += g
        if r0 <= a and b <= r1:
            for acc, g in zip(g_last, gs):
                acc += g
        logits.append(y.detach())
        loss += float(l.detach())
    drop = [g - gl for g, gl in zip(grads, g_last)]
    return dict(names=names, logits=torch.cat(logits), deformed=torch.cat(deformed) if deformed else None, loss=loss,
                grads=grads, drop=drop)


def entry_err(got, ref):
    """max |got - ref| / max |ref| (per entry, relative to the tensor's largest reference entry)."""
    d = float((got.double() - ref).abs().max())
    s = float(ref.abs().max())
    return d / s if s > 0 else d


def split_params(flat, names, ref_grads):
    out, off = [], 0
    for g in ref_grads:
        n = g.numel()
        out.append(flat[off:off + n].view(g.shape))
        off += n
    assert off == flat.numel()
    return out


def run_kernels(A, case, prior, params, spec, target, mode):
    """Logits, deformation, autograd gradients (``awb_prior_backward`` with dlogits of the same loss) and the loss and
    gradient of one fused step (Adam's first ``exp_avg`` is 0.1 g)."""
    N = spec.n_pixels
    Oo, P = params.shape
    ws = prior.new_workspace(N, A._lib.AWB_WS_TRAINING, DEV)
    want_deformed = case["kind"] == "flow" and mode == A._lib.AWB_FWD_EXACT_TRAINING
    logits, deformed = prior.forward(params, spec, mode, ws, want_deformed=want_deformed)
    s = torch.sigmoid(logits.double())
    dlog = (2.0 * (s - target.double()) * s * (1 - s) / N).float().contiguous()
    g_ag, _ = prior.backward(params, spec, dlog, ws, False)
    del ws
    f = A.PriorFitter(prior, params.detach().clone(), spec, target, A.LossConfig("mse"), A.OptimConfig("adam", lr=1e-3),
                      use_graph=False)
    loss = f.run(1)[0].double().cpu()
    g_fs = f.opt_state[:4 * Oo * P].view(torch.float32).view(Oo, P) * 10.0
    assert not f.scalars().nonfinite
    return logits, deformed, g_ag, loss, g_fs


# --------------------------------------------------------------------------------------------- exact fp32 path: the cases
def _case(id_, branch, kind, C_, F, B, H, W, expect, O_=1, flow_eval=1, L=2):
    return dict(id=id_, branch=branch, kind=kind, C=C_, F=F, L=L, B=B, H=H, W=W, O=O_, flow_eval=flow_eval,
                precision="fp32", expect=expect)


FP32_CASES = [
    # calibration: the regime the suite already covers (C = 2, 640x480: 148 ranges of 2080 rows, R = 2 + one remainder round)
    _case("calib", "C = 2 unit loops, 1 x 480 x 640 (tolerance calibration)", "flow", 2, 12, 1, 480, 640,
          {"bwd.kernel": "k_flow_bwd<2>", "bwd.dz_smem": True, "bwd.R": 2, "bwd.rounds1": 1}),
    # k_flow_bwd<3>: running gradient and pass partial in shared memory up to N = 571,872 (F = 18), in dX / flowd above
    _case("bwd3-smem-edge", "k_flow_bwd<3> shared-memory variant at its last N", "flow", 3, 18, 1, 736, 777,
          {"N": 571872, "bwd.kernel": "k_flow_bwd<3>", "bwd.dz_smem": True, "bwd.chunk": 3864}),
    _case("bwd3-global-edge", "k_flow_bwd<3> global-memory variant at its first N", "flow", 3, 18, 1, 1, 571873,
          {"N": 571873, "bwd.kernel": "k_flow_bwd<3>", "bwd.dz_smem": False, "bwd.chunk": 3872}),
    _case("configs4-loops", "configs[4] batch 2 x 480 x 640, global variant, unit-loop forward", "flow", 3, 18, 2, 480, 640,
          {"bwd.kernel": "k_flow_bwd<3>", "bwd.dz_smem": False, "bwd.chunk": 4152}),
    _case("configs4-tables", "configs[4] batch, global variant, segment-table forward (flow_eval 2)", "flow", 3, 18, 2, 480,
          640, {"bwd.kernel": "k_flow_bwd<3>", "bwd.dz_smem": False}, flow_eval=2),
    _case("bwd3-global-O4", "k_flow_bwd<3> global variant, 4 grouped objects ([O][N][4] offsets of flowd)", "flow", 3, 18, 1,
          600, 960, {"bwd.kernel": "k_flow_bwd<3>", "bwd.dz_smem": False}, O_=4),
    # k_flow_bwd<2> (unit loops): shared memory up to N = 2,610,720 (F = 12)
    _case("bwd2-smem-edge", "k_flow_bwd<2> shared-memory variant at its last N", "flow", 2, 12, 1, 1568, 1665,
          {"N": 2610720, "bwd.kernel": "k_flow_bwd<2>", "bwd.dz_smem": True}),
    _case("bwd2-global-edge", "k_flow_bwd<2> global-memory variant at its first N", "flow", 2, 12, 1, 1, 2610721,
          {"N": 2610721, "bwd.kernel": "k_flow_bwd<2>", "bwd.dz_smem": False}),
    # k_flow_bwd_seg<true / false> (C = 2 segment tables): 220 KiB reached at N = 647,648 (F = 12)
    _case("seg-smem-edge", "k_flow_bwd_seg<true> at its last N", "flow", 2, 12, 1, 592, 1094,
          {"N": 647648, "bwd.kernel": "k_flow_bwd_seg<true>"}, flow_eval=2),
    _case("seg-global-edge", "k_flow_bwd_seg<false> at its first N", "flow", 2, 12, 1, 747, 867,
          {"N": 647649, "bwd.kernel": "k_flow_bwd_seg<false>"}, flow_eval=2),
]
# small-N geometry, C = 2 and 3: (tag, B, H, W, branch, expected geometry)
SMALL = [
    ("n1", 1, 1, 1, "one pixel: one range, T = 32, forward chunk clamped to 32",
     {"N": 1, "bwd.S": 1, "bwd.T": 32, "bwd.R": 0, "bwd.rounds1": 1, "fwd.chunk": 32, "fwd.T": 32}),
    ("n31", 1, 1, 31, "one partial warp", {"N": 31, "bwd.T": 32, "fwd.chunk": 32, "fwd.S": 1}),
    ("n32", 1, 4, 8, "one full warp", {"N": 32, "bwd.chunk": 32, "bwd.T": 32, "fwd.S": 1}),
    ("n255", 1, 15, 17, "one range just below 256 rows", {"N": 255, "bwd.S": 1, "bwd.chunk": 256, "bwd.T": 256}),
    ("n257", 1, 1, 257, "two ranges of 136 and 121 rows, T = 160", {"N": 257, "bwd.S": 2, "bwd.chunk": 136, "bwd.T": 160}),
    ("n37887", 1, 173, 219, "148 ranges of 256 rows, the last one short",
     {"N": 37887, "bwd.S": 148, "bwd.chunk": 256, "bwd.empty": 0}),
    ("n37888", 1, 148, 256, "148 full ranges of 256 rows: R = 0, one remainder round",
     {"N": 37888, "bwd.chunk": 256, "bwd.empty": 0, "bwd.R": 0, "bwd.rounds1": 1}),
    ("n37889", 1, 1, 37889, "chunk rounded up to 264: ranges 144..147 empty (zero-partial exit)",
     {"N": 37889, "bwd.S": 148, "bwd.chunk": 264, "bwd.empty": 4}),
    ("r0", 1, 296, 384, "R = 0 with three remainder rounds", {"bwd.chunk": 768, "bwd.R": 0, "bwd.rounds1": 3, "bwd.empty": 0}),
    ("exact", 1, 296, 512, "chunk = one full round exactly: R = 1, no remainder round",
     {"bwd.chunk": 1024, "bwd.R": 1, "bwd.rounds1": 0, "bwd.empty": 0}),
    ("ragged-b3", 3, 17, 29, "three frames, odd sizes", {"N": 1479, "bwd.S": 6, "bwd.chunk": 248}),
]
for C_, F in ((2, 12), (3, 18)):
    for tag, B, H, W, branch, ex in SMALL:
        FP32_CASES.append(_case(f"c{C_}-{tag}", branch, "flow", C_, F, B, H, W, ex))
FP32_CASES.append(_case("c3-r1-remainder", "R = 2 plus one remainder round, C = 3", "flow", 3, 18, 1, 480, 640,
                        {"bwd.R": 2, "bwd.rounds1": 1, "bwd.dz_smem": True}))
FP32_CASES.append(_case("icnn-c3-n37889", "ICNN alone: empty trailing ranges of the exact path's reductions", "icnn", 3, 0, 1,
                        1, 37889, {"bwd.empty": 4}, L=1))


@pytest.mark.parametrize("case", FP32_CASES, ids=[c["id"] for c in FP32_CASES])
def test_exact_path_against_float64(A, case):
    """Exact fp32 path at one side of a launch branch: logits, loss, flow deformation and every parameter gradient (autograd
    backward and fused step) per entry against float64, with the tolerances of the calibration case; and the float64
    self-check that dropping the backward's last non-empty pixel range moves some gradient entry by more than TOL_GRAD."""
    r = check_regime(case)
    models = make_models(A, case)
    prior, params = make_handle(A, case, models)
    spec = grid_spec(A, case)
    target = make_target(case)
    logits, deformed, g_ag, loss, g_fs = run_kernels(A, case, prior, params, spec, target, A._lib.AWB_FWD_EXACT_TRAINING)
    rows = O.pixelize(torch_grid("linspace", case["B"], case["H"], case["W"], case["C"]))
    worst = dict(fwd=0.0, loss=0.0, grad=0.0, sens=float("inf"))
    for o, m in enumerate(models):
        ref = reference(m, case["kind"], rows, target[o], r["bwd.last"])
        worst["fwd"] = max(worst["fwd"], entry_err(logits[o], ref["logits"]))
        if ref["deformed"] is not None:
            worst["fwd"] = max(worst["fwd"], entry_err(deformed[o], ref["deformed"]))
        worst["loss"] = max(worst["loss"], abs(float(loss[o]) - ref["loss"]) / ref["loss"])
        errs = {}
        for src, flat in (("autograd", g_ag[o]), ("fused step", g_fs[o])):
            for k, g, g64 in zip(ref["names"], split_params(flat, ref["names"], ref["grads"]), ref["grads"]):
                errs[(src, k)] = entry_err(g, g64)
        sens = max(entry_err(gd, g64) for gd, g64 in zip(ref["drop"], ref["grads"]))
        worst["grad"] = max(worst["grad"], max(errs.values()))
        worst["sens"] = min(worst["sens"], sens)
        print(f"[regime {case['id']}] N={r['N']} object {o}: logits/deformation {worst['fwd']:.2e}  loss {worst['loss']:.2e}  "
              f"gradients {max(errs.values()):.2e} ({max(errs, key=errs.get)})  dropped-range {sens:.2e}")
        bad = {k: v for k, v in errs.items() if not v <= TOL_GRAD}
        assert not bad, f"{case['id']} object {o}: gradient entries off by more than {TOL_GRAD:g} of max: {bad}"
        assert sens > TOL_GRAD, f"{case['id']}: dropping rows {r['bwd.last']} moves no gradient by more than TOL_GRAD ({sens:.2e})"
    assert worst["fwd"] <= TOL_FWD, (case["id"], worst)
    assert worst["loss"] <= TOL_LOSS, (case["id"], worst)


# --------------------------------------------------------------------------------------------------------- tensor path
def _tc(id_, branch, kind, C_, L, B, H, W, expect, O_=1, F=12):
    return dict(id=id_, branch=branch, kind=kind, C=C_, F=F, L=L, B=B, H=H, W=W, O=O_, flow_eval=0, precision="f16",
                expect=expect)


TC_CASES = [
    _tc("icnn-c2-l1-n1", "one partial tile of one row", "icnn", 2, 1, 1, 1, 1, {"tc.n_tiles": 1, "tc.grid": 1, "tc.rem": 1}),
    _tc("icnn-c3-l2-n127", "one partial tile, N % 128 = 127", "icnn", 3, 2, 1, 1, 127, {"tc.n_tiles": 1, "tc.rem": 127}),
    _tc("icnn-c2-l2-n129", "a full tile and one row", "icnn", 2, 2, 1, 3, 43, {"tc.n_tiles": 2, "tc.grid": 2, "tc.rem": 1}),
    _tc("icnn-c3-l1-n129", "a full tile and one row, C = 3, three frames", "icnn", 3, 1, 3, 1, 43,
        {"tc.n_tiles": 2, "tc.rem": 1}),
    _tc("flow-c2-l2-n1", "flow prior, one pixel", "flow", 2, 2, 1, 1, 1, {"tc.n_tiles": 1}),
    _tc("flow-c3-l2-n127", "flow prior, N % 128 = 127", "flow", 3, 2, 1, 1, 127, {"tc.rem": 127}, F=18),
    _tc("icnn-c2-l2-148tiles", "n_tiles = CTA count (148), last tile 127 rows", "icnn", 2, 2, 1, 19, 997,
        {"tc.n_tiles": 148, "tc.grid": 148, "tc.rem": 127}),
    _tc("icnn-c3-l2-148tiles", "n_tiles = CTA count (148), no partial tile", "icnn", 3, 2, 1, 128, 148,
        {"tc.n_tiles": 148, "tc.grid": 148, "tc.rem": 0}),
    _tc("icnn-c2-l1-149tiles", "n_tiles = CTA count + 1, last tile one row", "icnn", 2, 1, 1, 45, 421,
        {"tc.n_tiles": 149, "tc.grid": 148, "tc.rem": 1}),
    _tc("icnn-c3-l2-149full", "n_tiles = CTA count + 1, all tiles full: CTA 0 takes a second full tile", "icnn", 3, 2, 1,
        149, 128, {"tc.n_tiles": 149, "tc.grid": 148, "tc.rem": 0}),
    _tc("flow-c2-l2-149tiles", "flow prior, n_tiles = CTA count + 1", "flow", 2, 2, 1, 149, 128,
        {"tc.n_tiles": 149, "tc.grid": 148}),
    _tc("flow-c3-l2-148tiles", "flow prior C = 3, n_tiles = CTA count", "flow", 3, 2, 2, 74, 128,
        {"tc.n_tiles": 148, "tc.grid": 148}, F=18),
    _tc("flow-c2-l2-o16-9tiles", "16 grouped objects: 9 CTAs each, n_tiles = 9", "flow", 2, 2, 1, 32, 36,
        {"tc.n_tiles": 9, "tc.grid": 9}, O_=16),
    _tc("icnn-c3-l1-o16-10tiles", "16 grouped objects, n_tiles = 10 (one CTA takes two tiles)", "icnn", 3, 1, 1, 1, 1153,
        {"tc.n_tiles": 10, "tc.grid": 9, "tc.rem": 1}, O_=16),
    _tc("icnn-c2-l1-o16-21tiles", "16 grouped objects, 2 or 3 tiles per CTA, the walk crosses rows and frames", "icnn", 2, 1,
        2, 23, 57, {"tc.n_tiles": 21, "tc.grid": 9, "tc.rem": 62}, O_=16),
    _tc("flow-c3-configs4", "configs[4]: 2 x 480 x 640, k_flow_bwd<3> global variant under the tensor path", "flow", 3, 2, 2,
        480, 640, {"tc.grid": 148, "bwd.kernel": "k_flow_bwd<3>", "bwd.dz_smem": False}, F=18),
]


@pytest.mark.parametrize("case", TC_CASES, ids=[c["id"] for c in TC_CASES])
def test_tensor_path_against_float64(A, case):
    """Tensor path (``k_icnn_fit_tc``) at the tile / CTA edges: fused-step loss against float64 within TC_TOL_LOSS (a dropped
    or doubled FULL tile moves the loss by about 1 / n_tiles; a partial last tile of a few rows by less, which is why the
    second-tile regime also has cases whose extra tiles are full), logits within the stated per-pixel bound, and the gradients
    of the fused step and of the autograd backward at the normwise bounds of DESIGN section 4: per tensor for the ICNN; for the
    flow, over its parameters as one block and per tensor against max(own norm, TC_FLOW_FLOOR x block norm)."""
    r = check_regime(case)
    models = make_models(A, case, seed=3)
    prior, params = make_handle(A, case, models)
    spec = grid_spec(A, case)
    target = make_target(case)
    logits, _, g_ag, loss, g_fs = run_kernels(A, case, prior, params, spec, target, A._lib.AWB_FWD_TC_TRAINING)
    rows = O.pixelize(torch_grid("linspace", case["B"], case["H"], case["W"], case["C"]))
    for o, m in enumerate(models):
        ref = reference(m, case["kind"], rows, target[o], r["bwd.last"])
        l_err = abs(float(loss[o]) - ref["loss"]) / ref["loss"]
        y_err = float(((logits[o].double() - ref["logits"]).abs() / ref["logits"].abs().clamp(min=1.0)).max())
        errs = {}
        for src, flat in (("autograd", g_ag[o]), ("fused step", g_fs[o])):
            flow = []
            for k, g, g64 in zip(ref["names"], split_params(flat, ref["names"], ref["grads"]), ref["grads"]):
                if k.startswith(("flow_net.", "linear.")):
                    flow.append((k, float((g.double() - g64).norm()), float(g64.norm())))
                elif float(g64.norm()) > 1e-7:
                    errs[(src, k)] = (float((g.double() - g64).norm() / g64.norm()), TC_TOL_GRAD_ICNN)
            if flow:
                block = sum(r_ ** 2 for _, _, r_ in flow) ** 0.5
                errs[(src, "flow_net + linear")] = (sum(d ** 2 for _, d, _ in flow) ** 0.5 / block, TC_TOL_GRAD_FLOW)
                for k, d, r_ in flow:
                    errs[(src, k)] = (d / max(r_, TC_FLOW_FLOOR * block), TC_TOL_GRAD_FLOW)
        worst = max(errs, key=lambda k: errs[k][0] / errs[k][1])
        print(f"[regime {case['id']}] N={r['N']} object {o}: loss {l_err:.2e}  logits {y_err:.2e}  "
              f"normwise gradients {errs[worst][0]:.2e} ({worst})")
        assert l_err <= TC_TOL_LOSS, (case["id"], o, l_err)
        assert y_err <= TC_LOGIT_BOUND, (case["id"], o, y_err)
        bad = {k: v for k, (v, tol) in errs.items() if not v <= tol}
        assert not bad, f"{case['id']} object {o}: normwise gradient errors above their bound: {bad}"


# ------------------------------------------------------------------------------------------ generated grid == explicit grid
GRID_CASES = [  # kind, precision, C, B, H, W
    ("icnn", "fp32", 3, 3, 1, 37), ("icnn", "fp32", 2, 1, 24, 1), ("icnn", "f16", 3, 3, 24, 1), ("icnn", "f16", 2, 1, 17, 30),
    ("flow", "fp32", 3, 3, 17, 30), ("flow", "fp32", 2, 1, 1, 64), ("flow", "f16", 3, 3, 9, 16), ("flow", "f16", 2, 3, 31, 1),
    ("icnn", "f16", 3, 1, 40, 56), ("flow", "f16", 3, 3, 33, 47),
]


def _grid_case(kind, precision, C_, B, H, W):
    return dict(id=f"{kind}-{precision}-c{C_}-{B}x{H}x{W}", kind=kind, precision=precision, C=C_, F=6 if C_ == 3 else 4, L=2,
                B=B, H=H, W=W, O=1, flow_eval=0)


@pytest.mark.parametrize("kind,precision,C_,B,H,W", GRID_CASES, ids=[_grid_case(*c)["id"] for c in GRID_CASES])
def test_generated_grid_equals_explicit_grid(A, kind, precision, C_, B, H, W):
    """linspace / index grids generated in the kernels == the same grid built by torch and passed explicitly: logits,
    autograd gradients, fused-step loss and gradient, bit for bit (``torch.equal``)."""
    case = _grid_case(kind, precision, C_, B, H, W)
    models = make_models(A, case, seed=5)
    prior, params = make_handle(A, case, models)
    target = make_target(case)
    fwd = A._lib.AWB_FWD_TC_TRAINING if precision == "f16" else A._lib.AWB_FWD_EXACT_TRAINING
    for mode in ("linspace", "index"):
        gen = run_kernels(A, case, prior, params, grid_spec(A, case, mode), target, fwd)
        exp = run_kernels(A, case, prior, params, A.GridSpecHost.from_tensor(torch_grid(mode, B, H, W, C_)), target, fwd)
        for name, a, b in zip(("logits", "deformation", "autograd gradients", "fused-step loss", "fused-step gradients"), gen, exp):
            if a is None:
                continue
            assert torch.equal(a, b), f"{mode}: {name} differ (max |d| {float((a - b).abs().max()):.3e})"


SLICE_WINDOWS = [(0, 1), (1, 421), (421, 1333), (1333, 1334), (1334, 2500), (2500, 2880)]     # frames of 960 rows, rows of 40


@pytest.mark.parametrize("kind,precision", [("icnn", "fp32"), ("icnn", "f16"), ("flow", "fp32"), ("flow", "f16")])
def test_slice_windows_generated_grid_equals_explicit_grid(A, kind, precision):
    """``slice_grads`` windows that start mid-frame and mid-row (every kernel walks the coordinates from ``row0``): the
    gradient rows of generated grids == those of the same grid built by torch, bit for bit, and they add up to the loss of
    the whole batch."""
    B, H, W, C_ = 3, 24, 40, 3
    case = dict(kind=kind, precision=precision, C=C_, F=6, L=2, B=B, H=H, W=W, O=1, flow_eval=0)
    models = make_models(A, case, seed=7)
    prior, params = make_handle(A, case, models)
    target = make_target(case)
    spec_loss = A.LossConfig("mse").to_specs(target)[0]
    ws = prior.new_workspace(max(e - b for b, e in SLICE_WINDOWS), A._lib.AWB_WS_FIT_STEP, DEV)
    for mode in ("linspace", "index"):
        rows = {}
        for key, spec in (("generated", grid_spec(A, case, mode)),
                          ("explicit", A.GridSpecHost.from_tensor(torch_grid(mode, B, H, W, C_)))):
            out = torch.empty((len(SLICE_WINDOWS), prior.grad_row_floats), dtype=torch.float32, device=DEV)
            for k, (b, e) in enumerate(SLICE_WINDOWS):
                prior.slice_grads(params, spec, b, e, target, spec_loss, out[k], ws)
            rows[key] = out
        assert torch.equal(rows["generated"], rows["explicit"]), \
            (mode, [k for k in range(len(SLICE_WINDOWS)) if not torch.equal(rows["generated"][k], rows["explicit"][k])])
        x = O.pixelize(torch_grid(mode, B, H, W, C_))
        ref = reference(models[0], kind, x, target[0], (0, 1))
        total = float(rows["generated"][:, -1].double().sum())
        assert abs(total - ref["loss"]) <= (TC_TOL_LOSS if precision == "f16" else TOL_LOSS) * ref["loss"], (mode, total, ref["loss"])


# ------------------------------------------------------------------------------- the tensor path's tile-to-tile coordinate walk
# k_icnn_fit_tc generates linspace coordinates by advancing a decomposed (frame, row, column) position by the CTA stride
# (gridDim.x * 128 rows) from tile to tile, with a column and a row carry.  That walk only runs when a CTA takes more than one
# tile; these shapes give every CTA several FULL tiles, a stride that is not a multiple of W (column carry) and batches of
# several frames (row carry into the frame), on ICNN priors (flow priors feed the kernel the flow's coordinates instead).
WALK_CASES = [  # C, L, B, H, W, O
    (2, 2, 3, 97, 101, 1), (3, 1, 3, 97, 101, 1), (3, 2, 3, 60, 77, 16), (2, 1, 2, 23, 57, 16),
]


def check_walk(n, H, W, O_, sms, row0=0):
    """Steps the walk of awb_tc_fit.cu (the position of every row of every CTA, advanced tile by tile) and counts the column
    and row carries taken on rows of FULL tiles past a CTA's first: the shape must make both happen."""
    grid = tc_geometry(n, O_, sms)["grid"]
    n_tiles, hw, d = cdiv(n, 128), H * W, grid * 128
    db, dr = divmod(d, hw)
    di, dj = divmod(dr, W)
    col = frame = 0
    for x in range(grid):
        for row in range(128):
            pb, r_ = divmod(row0 + x * 128 + row, hw)
            pi, pj = divmod(r_, W)
            for tile in range(x + grid, n_tiles, grid):
                pj += dj
                c1 = pj >= W
                if c1:
                    pj -= W
                    pi += 1
                pi += di
                c2 = pi >= H
                if c2:
                    pi -= H
                    pb += 1
                pb += db
                assert (pb, pi, pj) == (lambda q: (q // hw, q % hw // W, q % W))(row0 + tile * 128 + row)
                if tile * 128 + 127 < n:
                    col += c1
                    frame += c2
    assert col > 0 and frame > 0, (n, H, W, O_, col, frame)
    return col, frame


@pytest.mark.parametrize("C_,L,B,H,W,O_", WALK_CASES, ids=[f"c{c[0]}-l{c[1]}-{c[2]}x{c[3]}x{c[4]}-o{c[5]}" for c in WALK_CASES])
def test_tensor_path_tile_walk_equals_explicit_grid(A, C_, L, B, H, W, O_):
    """Tensor path, CTAs taking several tiles: the linspace coordinates the kernel walks from tile to tile == torch's grid
    passed explicitly (read per row, no walk), bit for bit in logits, autograd gradients, fused-step loss and gradient."""
    case = dict(id="walk", kind="icnn", precision="f16", C=C_, F=0, L=L, B=B, H=H, W=W, O=O_, flow_eval=0)
    check_walk(B * H * W, H, W, O_, torch.cuda.get_device_properties(0).multi_processor_count)
    models = make_models(A, case, seed=9)
    prior, params = make_handle(A, case, models)
    target = make_target(case)
    fwd = A._lib.AWB_FWD_TC_TRAINING
    gen = run_kernels(A, case, prior, params, grid_spec(A, case, "linspace"), target, fwd)
    exp = run_kernels(A, case, prior, params, A.GridSpecHost.from_tensor(torch_grid("linspace", B, H, W, C_)), target, fwd)
    for name, a, b in zip(("logits", "deformation", "autograd gradients", "fused-step loss", "fused-step gradients"), gen, exp):
        if a is None:
            continue
        assert torch.equal(a, b), f"{name} differ (max |d| {float((a - b).abs().max()):.3e})"


WALK_WINDOWS = [(0, 1234), (1234, 25000), (25000, 29391)]     # 3 x 97 x 101: the middle window starts mid-row (1234 = 12 x 101 + 22)


@pytest.mark.parametrize("C_", [2, 3])
def test_slice_window_tile_walk_equals_explicit_grid(A, C_):
    """``slice_grads`` on the tensor path with a window that starts mid-row and has more tiles than CTAs: the walk starts from
    ``row0`` and steps across rows and frames.  Gradient rows of the generated grid == those of torch's grid, bit for bit, and
    the rows add up to the float64 loss of the whole batch."""
    B, H, W = 3, 97, 101
    case = dict(kind="icnn", precision="f16", C=C_, F=0, L=2, B=B, H=H, W=W, O=1, flow_eval=0)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    b0, e0 = WALK_WINDOWS[1]
    assert b0 % W != 0
    check_walk(e0 - b0, H, W, 1, sms, row0=b0)
    models = make_models(A, case, seed=11)
    prior, params = make_handle(A, case, models)
    target = make_target(case)
    spec_loss = A.LossConfig("mse").to_specs(target)[0]
    ws = prior.new_workspace(max(e - b for b, e in WALK_WINDOWS), A._lib.AWB_WS_FIT_STEP, DEV)
    rows = {}
    for key, spec in (("generated", grid_spec(A, case, "linspace")),
                      ("explicit", A.GridSpecHost.from_tensor(torch_grid("linspace", B, H, W, C_)))):
        out = torch.empty((len(WALK_WINDOWS), prior.grad_row_floats), dtype=torch.float32, device=DEV)
        for k, (b, e) in enumerate(WALK_WINDOWS):
            prior.slice_grads(params, spec, b, e, target, spec_loss, out[k], ws)
        rows[key] = out
    assert torch.equal(rows["generated"], rows["explicit"]), \
        [k for k in range(len(WALK_WINDOWS)) if not torch.equal(rows["generated"][k], rows["explicit"][k])]
    ref = reference(models[0], "icnn", O.pixelize(torch_grid("linspace", B, H, W, C_)), target[0], (0, 1))
    total = float(rows["generated"][:, -1].double().sum())
    assert abs(total - ref["loss"]) <= TC_TOL_LOSS * ref["loss"], (total, ref["loss"])
