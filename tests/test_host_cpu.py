"""CPU-side checks: the C-ABI library loads and exports every symbol include/awb.h declares, the
drop-in modules keep the reference's state-dict contract, and nothing computes without a GPU."""
import os
import re

import pytest
import torch

import __graft_entry__ as entry

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module", autouse=True)
def built():
    entry.build()


def test_header_symbols_exported():
    from awesome_b200 import _lib
    lib = _lib.load()
    header = open(os.path.join(ROOT, "include", "awb.h")).read()
    declared = set(re.findall(r"\b(awb_[a-z_0-9]+)\s*\(", header))
    bound = {name for name, _, _ in _lib.SYMBOLS}
    assert declared == bound, f"header/binding mismatch: {declared ^ bound}"
    for name in declared:
        assert hasattr(lib, name)
    assert b"sm_100a" in lib.awb_version()


def test_header_constants_match_binding():
    from awesome_b200 import _lib
    header = open(os.path.join(ROOT, "include", "awb.h")).read()
    defined = {name: int(value) for name, value in
               re.findall(r"^#define\s+(AWB_[A-Z0-9_]+)\s+\(?(-?\d+)\)?(?:\s|$)", header, re.M)}
    assert {"AWB_WS_INFERENCE", "AWB_WS_SECOND_ORDER", "AWB_FWD_EXACT", "AWB_FWD_TC_TRAINING"} <= set(defined)
    for name, value in defined.items():
        if name.startswith(("AWB_WS_", "AWB_FWD_")):
            assert hasattr(_lib, name), f"{name} is not mirrored in _lib.py"
        if hasattr(_lib, name):
            assert getattr(_lib, name) == value, f"{name}: header {value}, _lib.py {getattr(_lib, name)}"


def test_state_dict_contract_matches_reference_fixture(golden):
    import awesome_b200 as A
    g = golden("icnn_c1.pt")
    m = A.ConvexNextNet(n_hidden_layers=1)
    sd = m.state_dict()
    assert list(sd.keys()) == list(g["init"].keys())
    for k in sd:
        assert sd[k].shape == g["init"][k].shape
    g2 = golden("icnn_c2.pt")
    m2 = A.ConvexNextNet(n_hidden=130, in_features=2, n_hidden_layers=2)
    assert list(m2.state_dict().keys()) == list(g2["init"].keys())
    m2.load_state_dict(g2["init"])
    # parameters stay views of one flat arena, in state_dict order
    off = m2._arena.data_ptr()
    for p in m2.parameters():
        assert p.data_ptr() == off
        off += 4 * p.numel()
    assert m2._arena.numel() == 35103
    cn = A.ConvexNet()
    assert list(cn.state_dict().keys()) == list(g2["convexnet_init"].keys())


def test_same_seed_same_init_as_reference(golden):
    import awesome_b200 as A
    g = golden("icnn_c1.pt")
    torch.manual_seed(0)
    m = A.ConvexNextNet(n_hidden_layers=1)
    for k, v in m.state_dict().items():
        assert torch.equal(v, g["init"][k]), k


def test_no_cpu_fallback():
    import awesome_b200 as A
    from awesome_b200._lib import AwbLibraryError
    m = A.ConvexNextNet()
    if not torch.cuda.is_available():
        with pytest.raises(AwbLibraryError):
            m(torch.zeros(1, 2, 4, 4))


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "awesome_b200")
    for dp, _, fns in os.walk(pkg):
        for fn in fns:
            if fn.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dp, fn)).read()
                for pat in ("import oracle", "from oracle", "oracle.", "oracle/"):
                    assert pat not in src, f"{fn} reaches into the oracle ({pat!r})"


def test_device_prior_cache_format_cpu():
    """DevicePriorCache keeps the reference PriorCache on-disk format (model_type, model_args, store_device, cache)."""
    import io
    import torch
    import awesome_b200 as A
    torch.manual_seed(0)
    c = A.DevicePriorCache(A.ConvexNextNet, dict(n_hidden_layers=2), capacity=1)
    m = A.ConvexNextNet(n_hidden_layers=2)
    c[3] = m.state_dict()
    c[5] = c.generate_prior(5)
    assert 3 in c and 5 in c and 4 not in c and len(c) == 2
    for k, v in m.state_dict().items():
        assert torch.equal(c[3][k], v)
    buf = io.BytesIO()
    c.save(buf)
    buf.seek(0)
    c2 = A.DevicePriorCache.load(buf)
    assert c2.model_type is A.ConvexNextNet and c2.model_args == dict(n_hidden_layers=2)
    m2 = A.ConvexNextNet(n_hidden_layers=2)
    c2.load_into(m2, 3)
    for a, b in zip(m2.state_dict().values(), m.state_dict().values()):
        assert torch.equal(a, b)


def test_fused_optimizer_delegates_non_arena_params_cpu():
    """Parameters outside a prior arena follow torch.optim exactly (the UNet side of a joint WrapperModule)."""
    import torch
    import awesome_b200 as A
    torch.manual_seed(0)
    a, b = torch.nn.Linear(5, 3), torch.nn.Linear(5, 3)
    b.load_state_dict(a.state_dict())
    oa, ob = A.FusedAdamax(a.parameters(), lr=1e-2, weight_decay=1e-3), torch.optim.Adamax(b.parameters(), lr=1e-2, weight_decay=1e-3)
    x = torch.randn(7, 5)
    for _ in range(3):
        for m, o in ((a, oa), (b, ob)):
            o.zero_grad()
            m(x).pow(2).sum().backward()
            o.step()
    for p, q in zip(a.parameters(), b.parameters()):
        assert torch.equal(p, q)


def test_multi_prior_container_keys_and_resize_cpu():
    import awesome_b200 as A
    m = A.NumberBasedMultiPriorModule(prior_type=A.ConvexNextNet, prior_args=dict(n_hidden_layers=1), min_priors=2)
    sd = m.state_dict()
    assert "priors.1.out.skp.weight" in sd and len({k.split(".")[1] for k in sd}) == 2
    big = A.NumberBasedMultiPriorModule(prior_type=A.ConvexNextNet, prior_args=dict(n_hidden_layers=1), min_priors=4)
    m.load_state_dict(big.state_dict())          # resizes like abstract_multi_prior_module.py:91-96
    assert len(m.priors) == 4


def test_diffeo_translate_keeps_arena_views_cpu():
    """ConvexDiffeomorphismNet.translate (reference :81-128): after the refit, `to` points land where `from` did."""
    import torch
    import awesome_b200 as A
    torch.manual_seed(0)
    m = A.ConvexDiffeomorphismNet()
    w0, b0 = m.linear.weight.detach().clone(), m.linear.bias.detach().clone()
    frm = torch.tensor([[0.2, 0.3], [0.7, 0.3], [0.2, 0.9]])
    to = frm + torch.tensor([0.1, -0.05])
    ptr = m.linear.weight.data_ptr()
    m.translate(frm, to)
    assert m.linear.weight.data_ptr() == ptr                      # still a view into the flat arena
    torch.testing.assert_close(to @ m.linear.weight.T + m.linear.bias, frm @ w0.T + b0, rtol=1e-4, atol=1e-5)
    assert [g for g in m._optimizer_group_ids()].count(3) == 4 * 2 * 2 + 4


def test_noisy_unaries_selection_cpu():
    """NoisyPathConnectedNet: round(T * p) frames, never the first / last, replaced once by clamp(randn + 0.5, 0, 1)."""
    import torch
    import awesome_b200 as A
    un = torch.rand(10, 6, 8)
    out, idx = A.noisy_unaries(un, 0.333, seed=0)
    assert len(idx) == 3 and 0 not in idx and 9 not in idx
    for i in range(10):
        assert torch.equal(out[i], un[i]) == (i not in idx)
    assert float(out.min()) >= 0.0 and float(out.max()) <= 1.0
    assert issubclass(A.NoisyPathConnectedNet, A.PathConnectedNet)
