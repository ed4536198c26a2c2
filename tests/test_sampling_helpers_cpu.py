"""``open_muse_b200.sampling`` (= ``muse.sampling`` of the drop-in package) against the reference module, function by function
on seeded inputs: the mask schedules of ``get_mask_chedule`` (the training masking rate and generate2's re-mask schedule),
``mask_by_random_topk`` through the same generator, ``top_k``, the Gumbel helpers.  What the reference returned (or raised)
is stored in tests/golden/ref_sampling.pt (make_golden.py::make_sampling)."""
import builtins

import pytest
import torch

import open_muse_b200.sampling as mine


@pytest.fixture(scope="module")
def ref(golden):
    return golden("ref_sampling.pt")


def test_public_names(ref):
    names = ref["public_names"]
    assert names and all(hasattr(mine, n) for n in names), [n for n in names if not hasattr(mine, n)]


@pytest.mark.parametrize("method", ["cosine", "linear", "sigmoid", "pow2", "pow3", "pow0.5", "pow", "log", "nonsense"])
def test_mask_schedules(ref, method):
    t, want = ref["schedule_t"], ref["schedules"][method]
    if isinstance(want, str):  # the reference raised this exception type
        with pytest.raises(getattr(builtins, want)):
            mine.get_mask_chedule(method)(t)
        return
    torch.testing.assert_close(mine.get_mask_chedule(method)(t), want, rtol=0, atol=0, equal_nan=True)


def test_sampling_helpers(ref):
    probs, x, t, want = ref["probs"], ref["x"], ref["t"], ref["outputs"]
    for temp, a in want["mask_by_random_topk"].items():
        b = mine.mask_by_random_topk(ref["mask_len"], probs, temperature=temp, generator=torch.Generator().manual_seed(1))
        assert torch.equal(a, b), temp
    assert torch.equal(want["top_k_07"], mine.top_k(x, 0.7)) and torch.equal(want["top_k"], mine.top_k(x))
    assert torch.equal(want["log"], mine.log(probs))
    assert torch.equal(want["gumbel_noise"], mine.gumbel_noise(probs, generator=torch.Generator().manual_seed(2)))
    assert torch.equal(want["gumbel_sample"], mine.gumbel_sample(x, temperature=0.5, generator=torch.Generator().manual_seed(3)))
    for fn, args in (("cosine_schedule", (t,)), ("linear_schedule", (t,)), ("sigmoid_schedule", (t,)), ("pow", (t, "pow2.5"))):
        torch.testing.assert_close(getattr(mine, fn)(*args), want[fn], rtol=0, atol=0)
