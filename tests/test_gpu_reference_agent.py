"""A ``PriorCache`` file written by the reference's ``PriorCache.save`` (stored fixture ``prior_cache_ref.pth``) loads
into ``DevicePriorCache`` and is written back in the same format."""
import torch


def test_reference_prior_cache_file_loads_into_device_cache(golden):
    """A file written by the reference's ``PriorCache.save`` (fixture ``prior_cache_ref.pth``, ``make_golden_full.py``) is the
    on-disk format ``DevicePriorCache`` reads and writes (``awesome/util/prior_cache.py:61-91``)."""
    import awesome_b200 as A
    state = golden("prior_cache_ref.pth")
    assert set(state) == {"model_type", "model_args", "store_device", "cache"} and set(state["cache"]) == {"0", "5"}
    cache = A.DevicePriorCache(A.ConvexNextNet, dict(n_hidden=130, in_features=2, n_hidden_layers=2), store_device=torch.device("cpu"))
    saved_type = state["model_type"]
    st = dict(state)
    st["model_type"] = "awesome_b200.ConvexNextNet"          # the YAML switch of INTEGRATION.md; keys and tensors untouched
    cache.set_state(st)
    assert 0 in cache and 5 in cache and 1 not in cache
    for key in (0, 5):
        got = cache[key]
        assert list(got.keys()) == list(state["cache"][str(key)].keys())
        for k, v in state["cache"][str(key)].items():
            assert torch.equal(got[k].cpu(), v), (key, k)
    back = cache.get_state()
    assert set(back) == set(state) and saved_type.endswith("ConvexNextNet")
    for k, v in state["cache"]["5"].items():
        assert torch.equal(back["cache"]["5"][k].cpu(), v)
