"""CPU-side checks of the drop-in F.grid_sample (rag_b200/grid_sample.py, csrc/grid_sample.cu): argument errors and workspace
queries of the C ABI without a GPU, the signature, the routing predicate's exclusions, and the install()/uninstall() binding
of F, alone and chained with resample=True."""
import inspect
import types

import pytest
import torch
import torch.nn.functional as F

FAKE = 256          # a 256-byte aligned non-null "pointer": every call below must fail before touching it


def test_exports_answer_errors_without_gpu():
    from rag_b200 import _cabi

    L = _cabi.lib()
    assert _cabi.ABI_VERSION == 17 and L.rag_abi_version() == 17
    fwd, bwd, ws = L.rag_grid_sample_fwd, L.rag_grid_sample_bwd, L.rag_grid_sample_bwd_workspace_bytes
    shape = (2, 3, 8, 16, 8, 16)
    # null pointers: -1
    assert fwd(None, FAKE, FAKE, *shape, 0, 0, None) == -1 and b"null" in L.rag_last_error()
    assert fwd(FAKE, None, FAKE, *shape, 0, 0, None) == -1
    assert fwd(FAKE, FAKE, None, *shape, 0, 0, None) == -1
    assert bwd(None, FAKE, FAKE, FAKE, FAKE, FAKE, 1 << 20, *shape, 0, 0, None) == -1
    assert bwd(FAKE, None, FAKE, None, FAKE, None, 0, *shape, 0, 0, None) == -1        # ggrid needs in
    assert bwd(FAKE, FAKE, FAKE, FAKE, None, None, 0, *shape, 0, 0, None) == -1        # gin needs the workspace
    # shapes: non-positive, and flat indices or the entry count reaching 2^31
    for bad in [(0, 3, 8, 16, 8, 16), (1, 3, 8, 16, 8, -1), (1, 1, 8, 16, 1 << 15, 1 << 14), (1, 1, 1 << 16, 1 << 15, 8, 8),
                (1, 64, 1 << 12, 1 << 13, 8, 8), (1, 64, 8, 8, 1 << 12, 1 << 13)]:
        assert fwd(FAKE, FAKE, FAKE, *bad, 0, 0, None) == -2, bad
        assert bwd(FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, 1 << 40, *bad, 0, 0, None) == -2, bad
        assert ws(*bad) == 0, bad
    assert fwd(FAKE, FAKE, FAKE, *shape, 2, 0, None) == -2 and b"padding_mode" in L.rag_last_error()   # reflection: not here
    # alignment: in / out 4 bytes, grid 8, workspace 256
    assert fwd(FAKE + 2, FAKE, FAKE, *shape, 0, 0, None) == -3
    assert fwd(FAKE, FAKE + 4, FAKE, *shape, 0, 1, None) == -3
    assert bwd(FAKE, FAKE, FAKE, FAKE, FAKE, FAKE + 16, 1 << 20, *shape, 1, 0, None) == -3
    # a workspace smaller than the query: -2, naming the query
    need = ws(*shape)
    assert bwd(FAKE, FAKE, FAKE, FAKE, None, FAKE, need - 1, *shape, 0, 0, None) == -2
    assert b"rag_grid_sample_bwd_workspace_bytes" in L.rag_last_error()


def test_workspace_query_needs_no_device():
    """20 bytes per sample-corner, 8 per input pixel, each region rounded up to 256 bytes, plus the sort's storage."""
    from rag_b200 import _cabi

    ws = _cabi.lib().rag_grid_sample_bwd_workspace_bytes
    up = lambda b: (b + 255) // 256 * 256            # noqa: E731
    for n, c, hi, wi, ho, wo in [(1, 1, 1, 1, 1, 1), (2, 3, 8, 16, 8, 16), (4, 3, 288, 576, 288, 576),
                                 (8, 3, 480, 960, 480, 960), (4, 32, 96, 192, 96, 192), (1, 3, 5, 7, 300, 2)]:
        m, p = 4 * n * ho * wo, n * hi * wi
        fixed = 5 * up(4 * m) + up(8 * p)
        got = ws(n, c, hi, wi, ho, wo)
        assert fixed < got <= fixed + 4 * 2**20, (n, c, hi, wi, ho, wo, got - fixed)
        assert ws(n, c + 5, hi, wi, ho, wo) == got                  # the channel count does not enter


def test_signature_is_f_grid_sample():
    from rag_b200 import grid_sample as G

    assert inspect.signature(G.grid_sample) == inspect.signature(F.grid_sample)
    base = types.SimpleNamespace(relu=F.relu, interpolate="base's interpolate")
    p = G.GridSampleProxy(base)
    assert p.grid_sample is G.grid_sample and p.relu is F.relu and p.interpolate == "base's interpolate"
    assert G.GridSampleProxy(F).avg_pool2d is F.avg_pool2d
    with pytest.raises(AttributeError):
        p.not_in_base


class _ReportsCuda(torch.Tensor):
    """A CPU tensor that answers is_cuda = True: lets the device-independent rest of the predicate be checked here."""

    @property
    def is_cuda(self):
        return True


def _cuda_like(*shape, dtype=torch.float32):
    return torch.zeros(*shape, dtype=dtype).as_subclass(_ReportsCuda)


def test_routing_positive_controls_and_exclusions():
    from rag_b200.grid_sample import routes

    x, g = _cuda_like(2, 3, 6, 8), _cuda_like(2, 5, 7, 2)
    # positive controls
    assert routes(x, g)
    assert routes(x, g, "bilinear", "border", True) and routes(x, g, "bilinear", "zeros", False)
    assert routes(_cuda_like(1, 1, 1, 1), _cuda_like(1, 1, 1, 2), align_corners=True)
    # each exclusion differs from a positive control in one argument
    excluded = {
        "CPU input": (torch.zeros(2, 3, 6, 8), g, {}),
        "CPU grid": (x, torch.zeros(2, 5, 7, 2), {}),
        "fp64 input": (_cuda_like(2, 3, 6, 8, dtype=torch.float64), g, {}),
        "fp64 grid": (x, _cuda_like(2, 5, 7, 2, dtype=torch.float64), {}),
        "fp16 input": (_cuda_like(2, 3, 6, 8, dtype=torch.float16), g, {}),
        "channels_last": (_cuda_like(2, 3, 6, 8).contiguous(memory_format=torch.channels_last), g, {}),
        "non-contiguous grid": (x, _cuda_like(2, 7, 5, 2).transpose(1, 2), {}),
        "nearest": (x, g, dict(mode="nearest")),
        "bicubic": (x, g, dict(mode="bicubic")),
        "reflection": (x, g, dict(padding_mode="reflection")),
        "5-D": (_cuda_like(2, 3, 4, 6, 8), _cuda_like(2, 3, 5, 7, 3), {}),
        "3-D grid": (x, _cuda_like(2, 35, 2), {}),
        "grid batch differs": (x, _cuda_like(1, 5, 7, 2), {}),
        "grid last axis not 2": (x, _cuda_like(2, 5, 7, 3), {}),
        "empty input": (_cuda_like(0, 3, 6, 8), _cuda_like(0, 5, 7, 2), {}),
        "no channels": (_cuda_like(2, 0, 6, 8), g, {}),
        "empty grid": (x, _cuda_like(2, 0, 7, 2), {}),
        "not tensors": ([[0.0]], g, {}),
    }
    for name, (xx, gg, kw) in excluded.items():
        assert not routes(xx, gg, **kw), name
    # out-of-limit sizes (too large to allocate here): the predicate's size test is the C library's
    from rag_b200.grid_sample import _within_limits

    assert _within_limits(1, 1, 2, 2, 1 << 14, 1 << 14) and not _within_limits(1, 1, 2, 2, 1 << 15, 1 << 14)   # 4*N*Ho*Wo
    assert not _within_limits(1, 64, 1 << 12, 1 << 13, 8, 8) and not _within_limits(1, 1, 1 << 16, 1 << 15, 8, 8)


def test_grid_sample_falls_through_on_cpu():
    from rag_b200.grid_sample import grid_sample

    gen = torch.Generator().manual_seed(0)
    x = torch.randn(2, 3, 5, 7, generator=gen)
    g = torch.rand(2, 4, 6, 2, generator=gen) * 2.2 - 1.1
    for kw in (dict(align_corners=True), dict(mode="nearest", align_corners=False), dict(padding_mode="reflection", align_corners=True)):
        assert torch.equal(grid_sample(x, g, **kw), F.grid_sample(x, g, **kw))
    with pytest.warns(UserWarning, match="align_corners=False"):
        assert torch.equal(grid_sample(x, g), F.grid_sample(x, g, align_corners=False))
    with pytest.raises(ValueError):          # F.grid_sample's own argument errors reach the caller
        grid_sample(x, g, mode="linear")


def _modules():
    from tests._mirror_net import reference_modules

    rag_model, mdenas, ops3d = reference_modules()
    rag_model.F = F
    loss = types.ModuleType("models.loss")
    loss.F = F
    cells = types.ModuleType("automl.build_model_2d")
    cells.F = F
    return rag_model, mdenas, ops3d, loss, cells


def test_install_binds_grid_sample_and_uninstall_restores():
    from rag_b200 import network as N
    from rag_b200.grid_sample import GridSampleProxy
    from rag_b200.grid_sample import grid_sample as ours

    rag_model, mdenas, ops3d, loss, cells = _modules()
    no_f = types.ModuleType("models.no_f")
    N.uninstall()
    try:
        with pytest.raises(ValueError, match="no_f"):
            N.install(rag_model, mdenas, ops3d, grid_sample=True, grid_sample_modules=(loss, no_f))
        assert loss.F is F                                     # nothing bound when one module is wrong
        with pytest.raises(ValueError, match="needs grid_sample_modules"):
            N.install(rag_model, mdenas, ops3d, grid_sample=True)
        done = N.install(None, None, None, grid_sample=True, grid_sample_modules=(loss,))
        assert done == {"models.loss": ["F.grid_sample"]}
        assert isinstance(loss.F, GridSampleProxy) and loss.F.base is F and loss.F.grid_sample is ours
        assert loss.F.avg_pool2d is F.avg_pool2d and loss.F.interpolate is F.interpolate
        # never wrapped twice
        N.install(None, None, None, grid_sample=True, grid_sample_modules=(loss, loss))
        assert loss.F.base is F
        # the flag off (modules given or not) binds nothing
        N.uninstall()
        N.install(rag_model, mdenas, ops3d, fuse_stem=True, grid_sample_modules=(loss,))
        assert loss.F is F and rag_model.F is F
    finally:
        N.uninstall()
    assert loss.F is F


@pytest.mark.parametrize("order", ["one call", "grid_sample first", "resample first"])
def test_grid_sample_chains_with_resample(order):
    from rag_b200 import network as N
    from rag_b200.grid_sample import GridSampleProxy
    from rag_b200.grid_sample import grid_sample as ours
    from rag_b200.resample import FProxy
    from rag_b200.resample import interpolate as our_interpolate

    rag_model, mdenas, ops3d, loss, cells = _modules()
    N.uninstall()
    try:
        gs = dict(grid_sample=True, grid_sample_modules=(loss,))
        rs = dict(resample=True, resample_modules=(loss, cells))
        if order == "one call":
            N.install(rag_model, mdenas, ops3d, **gs, **rs)
        else:
            first, second = (gs, rs) if order == "grid_sample first" else (rs, gs)
            N.install(rag_model, mdenas, ops3d, **first)
            N.install(rag_model, mdenas, ops3d, **second)
        assert isinstance(loss.F, GridSampleProxy) and isinstance(loss.F.base, FProxy)
        assert loss.F.grid_sample is ours and loss.F.interpolate is our_interpolate and loss.F.relu is F.relu
        assert isinstance(cells.F, FProxy) and isinstance(rag_model.F, FProxy)      # only the listed module gets grid_sample
        assert N.uninstall() > 0
    finally:
        N.uninstall()
    for m in (rag_model, loss, cells):
        assert m.F is F
