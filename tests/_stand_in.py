"""A stand-in with the growable network's structure (the reference's module layout: ``automl.operations_3d``,
``automl.build_model_3d``, ``models.rag_model``) and what it takes to check a training step of it on the kernels against a
plain reference of the same module tree:

* ``ref_forward``: feature -> ``oracle.cost_volume_ref`` -> matching -> ``oracle.disp_head_ref``, no ``install()``;
* ``ReluPins``: records each ReLU site's decision (``out > 0``) per call in one run and replays it in another, so that
  runs in different precisions are compared with the same ReLU decisions;
* ``Routes``: spies on the entry points of the hand-written layers, recording which layer and which resample took them.
"""
import types

import torch
import torch.nn as nn

from oracle import rag_oracle as O

_OPS_3D = '''
import torch.nn as nn
import torch.nn.functional as F


class ConvBR_3d(nn.Module):
    """The reference's field layout (operations_3d.py): .conv, .bn, .use_bn, .relu."""

    def __init__(self, c, o, k, s, p, bn=True, relu=True):
        super().__init__()
        self.conv = nn.Conv3d(c, o, k, stride=s, padding=p, bias=False)
        self.use_bn = bn
        self.bn = nn.BatchNorm3d(o) if bn else None
        self.relu = relu

    def forward(self, x):
        x = self.conv(x)
        if self.use_bn:
            x = self.bn(x)
        return F.relu(x, inplace=True) if self.relu else x
'''

_CELLS = '''
import torch
import torch.nn as nn
import torch.nn.functional as F


class Cell_2d(nn.Module):
    """Feature-Net cell: a level-3 and a level-6 branch joined by bilinear resampling."""

    def __init__(self, c):
        super().__init__()
        self.a = nn.Sequential(nn.Conv2d(c, c, 3, padding=1, bias=False), nn.BatchNorm2d(c), nn.ReLU())
        self.b = nn.Sequential(nn.Conv2d(c, c, 3, padding=1, bias=False), nn.BatchNorm2d(c), nn.ReLU())
        self.out = nn.Conv2d(2 * c, c, 1, bias=False)

    def forward(self, x):
        h, w = x.shape[2:]
        s0 = self.a(x)
        s1 = self.b(F.interpolate(s0, (h // 2, w // 2), mode="bilinear", align_corners=True))
        s1 = F.interpolate(s1, (h, w), mode="bilinear", align_corners=True)
        return self.out(torch.cat([s0, s0 + s1], 1))


class Cell_3d(nn.Module):
    """Matching-Net cell: a 1x1x1 preprocess, 3x3x3 ops, trilinear down- and up-sampling, step sums and a cat."""

    def __init__(self, c, k):
        super().__init__()
        self.pre = ConvBR_3d(c, k, 1, 1, 0)
        self.op0 = ConvBR_3d(k, k, 3, 1, 1)
        self.op1 = ConvBR_3d(k, k, 3, 1, 1)
        self.op2 = ConvBR_3d(k, k, 3, 1, 1)

    def forward(self, x):
        d, h, w = x.shape[2:]
        s0 = self.pre(x)
        s1 = self.op0(s0)
        low = self.op1(F.interpolate(s1, [d // 2, h // 2, w // 2], mode="trilinear", align_corners=True))
        s2 = self.op2(s0 + s1) + F.interpolate(low, [d, h, w], mode="trilinear", align_corners=True)
        return torch.cat([s0, s1, s2], 1), low
'''

_RAG_MODEL = '''
import torch.nn as nn
import torch.nn.functional as F


class Disp(nn.Module):
    def __init__(self, maxdisp):
        super().__init__()
        self.maxdisp = maxdisp


class DisparityRegression(nn.Module):
    pass


class Network(nn.Module):
    """The growable network's structure: feature net (stem + a 2-D cell), cost volume, matching net (stem3d0/1, a 3-D cell,
    last_6_3d, upsample_6, last_3_3d) and the head; forward / search_forward are bound by install().  With level12=True the
    matching net also has a level-12 branch: the cell's level-3 output down-sampled by 4, a last_12_3d-style pointwise layer
    and upsample_12 into last_6_3d's output."""

    def __init__(self, maxdisp=48, c=12, k=4, level12=False):
        super().__init__()
        self.maxdisp = maxdisp
        self.stem2d = nn.Sequential(nn.Conv2d(3, c, 3, stride=3, bias=False), nn.BatchNorm2d(c), nn.ReLU())
        self.cell2d = cells.Cell_2d(c)
        self.stem3d0 = ConvBR_3d(2 * c, c, 3, 1, 1)
        self.stem3d1 = ConvBR_3d(c, c, 3, 1, 1)
        self.cell3d = cells.Cell_3d(c, k)
        self.last_6_3d = ConvBR_3d(k, 3 * k, 1, 1, 0)
        self.last_3_3d = ConvBR_3d(3 * k, 1, 3, 1, 1, bn=False, relu=False)
        if level12:
            self.last_12_3d = ConvBR_3d(3 * k, 3 * k, 1, 1, 0)
        self.disp = Disp(maxdisp)

    def feature(self, x, task_arch=None, path=None):
        return self.cell2d(self.stem2d(x))

    def matching(self, cost, task_arch=None, path=None):
        x = self.stem3d1(self.stem3d0(cost))
        x3, x6 = self.cell3d(x)
        y6 = self.last_6_3d(x6)
        if hasattr(self, "last_12_3d"):
            d, h, w = x3.shape[2:]
            x12 = F.interpolate(x3, [d // 4, h // 4, w // 4], mode="trilinear", align_corners=True)
            upsample_12 = nn.Upsample(size=y6.size()[2:], mode="trilinear", align_corners=True)
            y6 = y6 + upsample_12(self.last_12_3d(x12))
        upsample_6 = nn.Upsample(size=x3.size()[2:], mode="trilinear", align_corners=True)
        return self.last_3_3d(x3 + upsample_6(y6))

    def forward(self, *a):
        raise NotImplementedError("bound by rag_b200.network.install")

    def search_forward(self, *a):
        raise NotImplementedError("bound by rag_b200.network.install")
'''


def _module(name, src, **inject):
    m = types.ModuleType(name)
    m.__dict__.update(inject)
    exec(compile(src, f"<stand-in {name}>", "exec"), m.__dict__)
    return m


def _stand_in():
    """Fresh module objects (rag_model, operations_3d, build_model_3d): an install() into one stand-in leaves another plain."""
    ops3d = _module("automl.operations_3d", _OPS_3D)
    cells = _module("automl.build_model_3d", _CELLS, ConvBR_3d=ops3d.ConvBR_3d)
    rag_model = _module("models.rag_model", _RAG_MODEL, ConvBR_3d=ops3d.ConvBR_3d, cells=cells)
    return rag_model, ops3d, cells


def ref_forward(net, left, right):
    """The plain forward of the stand-in, in the dtype and on the device of ``net``: what ``install()``'s network_forward
    computes, with the oracle's cost volume and head."""
    x, y = net.feature(left), net.feature(right)
    return O.disp_head_ref(net.matching(O.cost_volume_ref(x, y, net.maxdisp)), net.maxdisp)


def _is_convbr(m):
    return type(m).__name__ == "ConvBR_3d"


def relu_sites(net):
    """Names of the modules whose output passes a ReLU: every ConvBR_3d with relu=True and every nn.ReLU."""
    return [n for n, m in net.named_modules() if isinstance(m, nn.ReLU) or (_is_convbr(m) and m.relu)]


class ReluPins:
    """The ReLU decisions of one run, per site and call, to replay in another run of the same module tree.

    ``record(net)`` keeps ``out > 0`` of every ReLU site of ``net`` (forward hooks, which also fire for a forward that
    ``install()`` rebound).  ``replay(net, ops3d)`` makes every site of ``net`` compute ``pre * mask`` with the recorded mask
    of the same call instead of ``relu(pre)`` -- ConvBR_3d.forward of the stand-in's ``ops3d`` rebound to conv -> bn -> mask,
    nn.ReLU hooks returning ``input * mask`` -- and keeps each pre-activation for ``flips``.  Both are context managers."""

    def __init__(self):
        self.masks = {}         # site name -> [mask of call 0, call 1, ...]
        self.pre = {}           # site name -> [pre-activation of call 0, ...] of the replaying run

    def record(self, net):
        sites = set(relu_sites(net))
        self.masks = {n: [] for n in sites}

        def hook(name):
            def fn(m, args, out):
                self.masks[name].append(out.detach() > 0)
            return fn

        return _Hooks([m.register_forward_hook(hook(n)) for n, m in net.named_modules() if n in sites])

    def replay(self, net, ops3d):
        names = {m: n for n, m in net.named_modules()}
        self.pre = {n: [] for n in self.masks}
        pins = self

        def mask(name, pre):
            k = len(pins.pre[name])
            pins.pre[name].append(pre.detach())
            return pins.masks[name][k].to(pre.dtype)

        def pinned_forward(self, x):
            x = self.conv(x)
            if self.use_bn:
                x = self.bn(x)
            return x * mask(names[self], x) if self.relu else x

        def relu_hook(m, args, out):
            return args[0] * mask(names[m], args[0])

        old = ops3d.ConvBR_3d.forward
        ops3d.ConvBR_3d.forward = pinned_forward
        handles = [m.register_forward_hook(relu_hook) for m in net.modules() if isinstance(m, nn.ReLU)]
        return _Hooks(handles, lambda: setattr(ops3d.ConvBR_3d, "forward", old))

    def calls(self):
        return sum(len(v) for v in self.masks.values())

    def flips(self, rel=1e-5):
        """How many replayed decisions the replaying run's own pre-activation contradicts (``(pre > 0) != mask``); asserts
        every one of them is rounding noise, |pre| <= rel * max |pre| of that call."""
        n = 0
        for name, pres in self.pre.items():
            assert len(pres) == len(self.masks[name]), f"{name}: {len(pres)} replayed calls of {len(self.masks[name])} recorded"
            for pre, m in zip(pres, self.masks[name]):
                f = (pre > 0) != m
                if f.any():
                    worst = (pre[f].abs().max() / pre.abs().max()).item()
                    assert worst <= rel, f"{name}: a ReLU decision differs beyond rounding noise (|pre| = {worst:.2e} of the max)"
                    n += int(f.sum())
        return n


class _Hooks:
    def __init__(self, handles, undo=None):
        self.handles, self.undo = handles, undo

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        for h in self.handles:
            h.remove()
        if self.undo is not None:
            self.undo()


# (module, attribute) of each hand-written path's entry point.  The routing code looks each of them up by name at call time,
# so a monkeypatched spy sees every call.  For the ConvBR_3d kinds the spy records the layer (the first argument) or the
# layer owning the weight argument; for the resamples, the kernel launched and the sizes.
ROUTES = {
    "stem": ("rag_b200.fused_stem", "cv_stem_forward"),               # (x, y, weight, ...): fused stem, FusedStemFn and inference
    "matching": ("rag_b200.matching_conv", "convbr_forward"),         # (layer, x): 3x3x3 ConvBR_3d, ConvBR3dFn and inference
    "pointwise": ("rag_b200.pointwise_conv", "convbr_forward"),       # (layer, x): 1x1x1 ConvBR_3d, PointwiseBR3dFn and inference
    "last_conv": ("rag_b200.last_conv", "conv3d_c1_forward"),         # (x, weight): last_3_3d, Conv3dC1Fn and inference
    "trilinear": ("rag_b200.upsample", "_resize"),                    # (kernel, src, dst shape, in size, out size, ...)
    "bilinear": ("rag_b200.resample", "_resize"),
}
# the autograd function each ConvBR_3d path runs when a gradient is wanted
AUTOGRAD = {"stem": "FusedStemFn", "matching": "ConvBR3dFn", "pointwise": "PointwiseBR3dFn", "last_conv": "Conv3dC1Fn"}
# where the routing code calls each entry point by name
CALLERS = {
    "stem": [("rag_b200.fused_stem", "stem_forward"), ("rag_b200.fused_stem", "FusedStemFn.forward")],
    "matching": [("rag_b200.matching_conv", "matching_forward")],
    "pointwise": [("rag_b200.pointwise_conv", "pointwise_forward")],
    "last_conv": [("rag_b200.last_conv", "conv_forward"), ("rag_b200.last_conv", "Conv3dC1Fn.forward")],
    "trilinear": [("rag_b200.upsample", "TrilinearResizeFn.forward"), ("rag_b200.upsample", "TrilinearResizeFn.backward")],
    "bilinear": [("rag_b200.resample", "BilinearResizeFn.forward"), ("rag_b200.resample", "BilinearResizeFn.backward")],
}


class Routes:
    """Spies on ``ROUTES`` (installed with pytest's ``monkeypatch``).  ``layers[name]`` is the set of paths the ConvBR_3d
    called ``name`` took; ``resizes`` lists (kernel, in size, out size) per resample launch."""

    def __init__(self, monkeypatch, net):
        import importlib

        self.layers, self.resizes = {}, []
        owner = {m.conv.weight: n for n, m in net.named_modules() if _is_convbr(m)}
        by_ptr = lambda w: next(n for p, n in owner.items() if p.data_ptr() == w.data_ptr())   # noqa: E731
        layer_name = {m: n for n, m in net.named_modules()}
        for path, (mod, attr) in ROUTES.items():
            mod = importlib.import_module(mod)
            orig = getattr(mod, attr)
            if path in ("trilinear", "bilinear"):
                def spy(fn_name, src, dst_shape, in_size, out_size, *a, _orig=orig):
                    self.resizes.append((fn_name, tuple(in_size), tuple(out_size)))
                    return _orig(fn_name, src, dst_shape, in_size, out_size, *a)
            else:
                def spy(*a, _orig=orig, _path=path, **k):
                    if _path in ("matching", "pointwise"):
                        name = layer_name[a[0]]
                    else:
                        name = by_ptr(a[2] if _path == "stem" else a[1])
                    self.layers.setdefault(name, set()).add(_path)
                    return _orig(*a, **k)
            monkeypatch.setattr(mod, attr, spy)
