"""CPU-side checks of the drop-in F.interpolate (rag_b200/resample.py, csrc/trilinear.cu's bilinear exports): argument errors
of the C ABI without a GPU, the signature, the routing predicate's exclusions, the output-size computation against
F.interpolate, and the install()/uninstall() binding of F."""
import inspect
import itertools
import types

import pytest
import torch
import torch.nn.functional as F

from tests._mirror_net import reference_modules

FAKE = 256          # a 16-byte aligned non-null "pointer": every call below must fail before touching it


def test_exports_answer_errors_without_gpu():
    from rag_b200 import _cabi

    L = _cabi.lib()
    assert _cabi.ABI_VERSION == 18 and L.rag_abi_version() == 18
    for fn in (L.rag_bilinear_resize_fwd, L.rag_bilinear_resize_bwd):
        # null pointers: -1 with "null" in the text
        assert fn(None, FAKE, 1, 4, 8, 8, 16, 1, None) == -1
        assert b"null" in L.rag_last_error() and b"bilinear_resize" in L.rag_last_error()
        assert fn(FAKE, None, 1, 4, 8, 8, 16, 0, None) == -1
        # shapes outside check_tri's limits: -2, before any pointer is touched
        for bc, hi, wi, ho, wo in [(0, 4, 8, 8, 16), (1, 0, 8, 8, 16), (1, 4, 8, 8, -1), (1, 4, 8, 10000, 12000),
                                   (1, 4, 8, 1, 21000)]:
            assert fn(FAKE, FAKE, bc, hi, wi, ho, wo, 1, None) == -2, (bc, hi, wi, ho, wo)
        # pointers not 4-byte aligned: -3
        assert fn(FAKE + 2, FAKE, 1, 4, 8, 8, 16, 1, None) == -3
        assert fn(FAKE, FAKE + 1, 1, 4, 8, 8, 16, 1, None) == -3


def test_signature_is_f_interpolate():
    from rag_b200 import resample

    assert inspect.signature(resample.interpolate) == inspect.signature(F.interpolate)
    assert resample.FProxy().interpolate is resample.interpolate
    assert resample.FProxy().relu is F.relu and resample.FProxy().smooth_l1_loss is F.smooth_l1_loss


class _ReportsCuda(torch.Tensor):
    """A CPU tensor that answers is_cuda = True: lets the device-independent rest of the predicate be checked here."""

    @property
    def is_cuda(self):
        return True


def _cuda_like(*shape, dtype=torch.float32):
    return torch.zeros(*shape, dtype=dtype).as_subclass(_ReportsCuda)


def test_routing_positive_controls_and_exclusions():
    from rag_b200.resample import plan

    x5, x4 = _cuda_like(2, 3, 4, 6, 8), _cuda_like(2, 3, 6, 8)
    # positive controls: the cells' calls and the other accepted forms
    assert plan(x5, size=(8, 12, 16), mode="trilinear", align_corners=True) == ((8, 12, 16), True)
    assert plan(x5, size=(2, 3, 4), mode="trilinear", align_corners=False) == ((2, 3, 4), False)
    assert plan(x5, size=5, mode="trilinear") == ((5, 5, 5), False)
    assert plan(x4, size=[12, 16], mode="bilinear", align_corners=True) == ((12, 16), True)
    assert plan(x4, scale_factor=2, mode="bilinear", align_corners=True) == ((12, 16), True)
    assert plan(x4, scale_factor=0.5, mode="bilinear", recompute_scale_factor=True) == ((3, 4), False)
    assert plan(x5, scale_factor=(2, 0.5, 1.5), mode="trilinear", align_corners=True) == ((8, 3, 12), True)
    # each exclusion differs from a positive control in one argument
    excluded = {
        "CPU tensor": (torch.zeros(2, 3, 6, 8), dict(size=(12, 16), mode="bilinear", align_corners=True)),
        "fp64": (_cuda_like(2, 3, 6, 8, dtype=torch.float64), dict(size=(12, 16), mode="bilinear", align_corners=True)),
        "channels_last": (_cuda_like(2, 3, 6, 8).contiguous(memory_format=torch.channels_last),
                          dict(size=(12, 16), mode="bilinear", align_corners=True)),
        "nearest": (x4, dict(size=(12, 16), mode="nearest")),
        "bicubic": (x4, dict(size=(12, 16), mode="bicubic", align_corners=True)),
        "area": (x4, dict(size=(12, 16), mode="area")),
        "linear": (_cuda_like(2, 3, 8), dict(size=16, mode="linear", align_corners=True)),
        "antialias": (x4, dict(size=(12, 16), mode="bilinear", align_corners=True, antialias=True)),
        "scale_factor, align_corners=False": (x4, dict(scale_factor=2, mode="bilinear", align_corners=False)),
        "scale_factor, align_corners=None": (x5, dict(scale_factor=2, mode="trilinear")),
        "3-D tensor": (_cuda_like(2, 3, 8), dict(size=16, mode="bilinear", align_corners=True)),
        "bilinear on 5-D": (x5, dict(size=(8, 12, 16), mode="bilinear", align_corners=True)),
        "trilinear on 4-D": (x4, dict(size=(12, 16), mode="trilinear", align_corners=True)),
        "empty tensor": (_cuda_like(0, 3, 6, 8), dict(size=(12, 16), mode="bilinear", align_corners=True)),
        "empty output": (x4, dict(size=(0, 16), mode="bilinear", align_corners=True)),
        "size and scale_factor": (x4, dict(size=(12, 16), scale_factor=2, mode="bilinear", align_corners=True)),
        "size of the wrong length": (x4, dict(size=(12, 16, 4), mode="bilinear", align_corners=True)),
        "non-integer size": (x4, dict(size=(12.0, 16), mode="bilinear", align_corners=True)),
        "axes too long for the tables": (x4, dict(size=(8, 30000), mode="bilinear", align_corners=True)),
    }
    for name, (x, kw) in excluded.items():
        assert plan(x, **kw) is None, name


def test_output_size_matches_f_interpolate():
    from rag_b200.resample import output_size

    n = 0
    for shape in [(1, 1, 5, 7), (1, 2, 3, 4, 9), (1, 1, 1, 13), (1, 1, 7, 1, 3)]:
        x = torch.zeros(shape)
        mode = "bilinear" if x.dim() == 4 else "trilinear"
        k = x.dim() - 2
        for s in [1, 2, 3, 8, 17]:
            size = tuple(s + i for i in range(k))
            assert output_size(x, size=size) == tuple(F.interpolate(x, size=size, mode=mode, align_corners=True).shape[2:])
            assert output_size(x, size=s) == tuple(F.interpolate(x, size=s, mode=mode, align_corners=True).shape[2:])
            n += 2
        for sf, ac, rc in itertools.product([0.5, 1 / 3, 0.7, 1.0, 1.5, 2, 2.5, 3, 4, 0.26], [True, False], [None, True]):
            for f in (sf, tuple(sf * (1 + 0.5 * i) for i in range(k))):
                got = output_size(x, scale_factor=f, recompute_scale_factor=rc)
                try:
                    want = tuple(F.interpolate(x, scale_factor=f, mode=mode, align_corners=ac, recompute_scale_factor=rc).shape[2:])
                except RuntimeError:             # an empty output axis: F.interpolate raises, the routing refuses it
                    assert min(got) <= 0, (shape, f)
                    continue
                assert got == want, (shape, f, ac, rc)
                n += 1
    assert n > 100


def test_interpolate_falls_through_on_cpu():
    from rag_b200.resample import interpolate

    x = torch.randn(2, 3, 5, 7, generator=torch.Generator().manual_seed(0))
    for kw in (dict(size=(9, 4), mode="bilinear", align_corners=True), dict(scale_factor=2, mode="nearest"),
               dict(scale_factor=0.5, mode="bilinear", align_corners=False)):
        assert torch.equal(interpolate(x, **kw), F.interpolate(x, **kw))
    with pytest.raises(ValueError):          # F.interpolate's own argument errors reach the caller
        interpolate(x, size=(9, 4), scale_factor=2, mode="bilinear")


def _stand_ins():
    rag_model, mdenas, ops3d = reference_modules()
    rag_model.F = F                          # the reference's `import torch.nn.functional as F`
    cells_2d = types.ModuleType("automl.build_model_2d")
    cells_2d.F = F
    cells_3d = types.ModuleType("automl.build_model_3d")
    cells_3d.F = F
    return rag_model, mdenas, ops3d, cells_2d, cells_3d


def test_install_binds_f_and_uninstall_restores():
    from rag_b200 import network as N
    from rag_b200.resample import FProxy
    from rag_b200.upsample import NNProxy

    rag_model, mdenas, ops3d, cells_2d, cells_3d = _stand_ins()
    no_f = types.ModuleType("automl.genotypes_2d")
    N.uninstall()
    with pytest.raises(ValueError, match="genotypes_2d"):
        N.install(rag_model, mdenas, ops3d, resample=True, resample_modules=(cells_2d, no_f))
    assert rag_model.F is F and cells_2d.F is F            # nothing bound when one module is wrong
    N.uninstall()
    with pytest.raises(ValueError, match="needs rag_model or resample_modules"):
        N.install(None, mdenas, ops3d, resample=True)
    N.uninstall()
    try:
        done = N.install(rag_model, mdenas, ops3d, fuse_stem=True, upsample=True, matching_convs=True, pointwise_convs=True,
                         resample=True, resample_modules=(cells_2d, cells_3d))
        for m in (rag_model, cells_2d, cells_3d):
            assert isinstance(m.F, FProxy)
        assert "F.interpolate" in done["rag_model"] and "nn.Upsample" in done["rag_model"]
        assert done["automl.build_model_2d"] == ["F.interpolate"] and done["automl.build_model_3d"] == ["F.interpolate"]
        assert isinstance(rag_model.nn, NNProxy)
        # resample_modules alone, without rag_model
        N.uninstall()
        N.install(None, None, None, resample=True, resample_modules=(cells_3d,))
        assert isinstance(cells_3d.F, FProxy) and rag_model.F is F
    finally:
        N.uninstall()
    for m in (rag_model, cells_2d, cells_3d):
        assert m.F is F


def test_resample_flag_off_changes_nothing():
    from rag_b200 import network as N

    rag_model, mdenas, ops3d, cells_2d, cells_3d = _stand_ins()
    flags = dict(fuse_stem=True, upsample=True, matching_convs=True, pointwise_convs=True)

    def snapshot():                          # every binding install() made; its proxies are fresh objects per call
        return {k: (type(getattr(*k)) if type(getattr(*k)).__name__.endswith("Proxy") else getattr(*k)) for k in N._ORIGINALS}

    N.uninstall()
    try:
        done_off = N.install(rag_model, mdenas, ops3d, **flags)
        bound_off = snapshot()
        assert rag_model.F is F and cells_2d.F is F
        N.uninstall()
        done_mods = N.install(rag_model, mdenas, ops3d, resample_modules=(cells_2d, cells_3d), **flags)   # modules, flag off
        assert rag_model.F is F and cells_2d.F is F and cells_3d.F is F
        assert done_mods == done_off and snapshot() == bound_off
        N.uninstall()
        N.install(rag_model, mdenas, ops3d, resample=True, resample_modules=(cells_2d,), **flags)
        on = snapshot()
        assert {k: v for k, v in on.items() if k[1] != "F"} == bound_off      # the other bindings are the flag-off ones
        assert {k[0] for k in on if k[1] == "F"} == {rag_model, cells_2d}
    finally:
        N.uninstall()
