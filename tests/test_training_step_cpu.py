"""Self-checks, without a GPU, of the harness tests/test_training_step_gpu.py compares a training step with: the plain
reference forward, the ReLU pins and the routing spies of tests/_stand_in.py."""
import importlib
import inspect

import pytest
import torch

from tests._stand_in import AUTOGRAD, CALLERS, ROUTES, ReluPins, _stand_in, ref_forward, relu_sites
from tests._util import gen, randn, sparse_grad


def _step(net, batches):
    for left, right, gpred in batches:
        pred = ref_forward(net, left, right)
        pred.backward(gpred)
    return pred.detach(), {n: p.grad.clone() for n, p in net.named_parameters()}, {n: b.clone() for n, b in net.named_buffers()}


@pytest.mark.parametrize("k, b, steps", [(4, 2, 1), (8, 1, 1), (4, 3, 2)])
def test_pinned_reference_reproduces_the_unpinned_run(k, b, steps):
    """Masks recorded from the plain fp64 run itself, replayed: the same prediction, gradients and running statistics,
    exactly, and no decision the replaying run's pre-activations contradict."""
    rag_model, ops3d, _ = _stand_in()
    g = gen(40 + k + b)
    torch.manual_seed(41)
    net = rag_model.Network(48, k=k, level12=True).double().train()
    state = {n: v.clone() for n, v in net.state_dict().items()}
    batches = [(randn((b, 3, 48, 96), g).double(), randn((b, 3, 48, 96), g).double(), sparse_grad((b, 48, 96), g, 0.7).double())
               for _ in range(steps)]
    pins = ReluPins()
    with pins.record(net):
        unpinned = _step(net, batches)
    plain_forward = ops3d.ConvBR_3d.forward
    net.load_state_dict(state)
    net.zero_grad(set_to_none=True)
    with pins.replay(net, ops3d):
        assert ops3d.ConvBR_3d.forward is not plain_forward
        pinned = _step(net, batches)
    assert ops3d.ConvBR_3d.forward is plain_forward
    assert all(not m._forward_hooks for m in net.modules())
    assert pins.flips() == 0
    assert torch.equal(unpinned[0], pinned[0])
    for a, b_ in zip(unpinned[1:], pinned[1:]):
        assert list(a) == list(b_) and all(torch.equal(a[n], b_[n]) for n in a), [n for n in a if not torch.equal(a[n], b_[n])]
    assert all(bool((unpinned[1][n] != 0).any()) for n in unpinned[1]), "a parameter without gradient"


def test_pins_catch_a_decision_beyond_rounding_noise():
    """A replayed mask that contradicts a pre-activation far from 0 fails ``flips``; one at rounding noise is counted."""
    pins = ReluPins()
    pins.masks = {"a": [torch.tensor([True, False, True])]}
    pins.pre = {"a": [torch.tensor([1.0, 1e-7, 2.0], dtype=torch.float64)]}
    assert pins.flips() == 1
    pins.pre = {"a": [torch.tensor([1.0, 0.5, 2.0], dtype=torch.float64)]}
    with pytest.raises(AssertionError, match="rounding noise"):
        pins.flips()


@pytest.mark.parametrize("k, level12", [(4, False), (4, True), (8, True)])
def test_recorder_captures_every_relu_site(k, level12):
    """3 nn.ReLU in the Feature Net, called once per image (twice per step); 7 ConvBR_3d with relu=True (8 with the
    level-12 branch), once per step; last_3_3d has no ReLU."""
    rag_model, _, _ = _stand_in()
    torch.manual_seed(0)
    net = rag_model.Network(48, k=k, level12=level12).double()
    g = gen(2)
    relus = ["stem2d.2", "cell2d.a.2", "cell2d.b.2"]
    convs = ["stem3d0", "stem3d1", "cell3d.pre", "cell3d.op0", "cell3d.op1", "cell3d.op2", "last_6_3d"] + (["last_12_3d"] if level12 else [])
    assert sorted(relu_sites(net)) == sorted(relus + convs)
    pins = ReluPins()
    with pins.record(net), torch.no_grad():
        for _ in range(2):
            ref_forward(net, randn((2, 3, 24, 48), g).double(), randn((2, 3, 24, 48), g).double())
    assert {n: len(v) for n, v in pins.masks.items()} == {**{n: 4 for n in relus}, **{n: 2 for n in convs}}
    assert pins.calls() == 2 * (2 * len(relus) + len(convs))
    assert pins.masks["stem3d0"][0].shape == (2, 12, 16, 8, 16) and pins.masks["stem2d.2"][0].dtype == torch.bool


def test_spies_wrap_functions_that_exist():
    """Every spied entry point exists, and the routing code looks it up by name at call time (so a monkeypatched spy sees
    every call): a rename fails here rather than silently on the GPU."""
    for path, (mod, attr) in ROUTES.items():
        assert callable(getattr(importlib.import_module(mod), attr)), (path, mod, attr)
        for cmod, cname in CALLERS[path]:
            fn = importlib.import_module(cmod)
            for part in cname.split("."):
                fn = getattr(fn, part)
            assert attr in inspect.unwrap(fn).__code__.co_names, f"{cmod}.{cname} does not call {attr} by name"
    for path, fn in AUTOGRAD.items():
        mod = importlib.import_module(ROUTES[path][0])
        assert issubclass(getattr(mod, fn), torch.autograd.Function), (path, fn)
