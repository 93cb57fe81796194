"""Drop-in boundary for the reference's stereo networks (SURVEY.md section 8 N-0).

The reference builds the cost volume inline in three ``forward`` methods and owns its ``Disp`` head:

* ``Network.forward(left, right, t, task_arch=None, path=None)``      src/models/rag_model.py:369-387
* ``Network.search_forward(left, right, t, selected_ops)``            src/models/rag_model.py:688-706
* ``BasicNetwork.forward(left, right, fea_ops, mat_ops)``             src/automl/mdenas_basicmodel.py:76-97

The functions below are those three methods with the nine inline cost-volume lines replaced by one
call to the CUDA kernel and ``self.disp`` routed through the fused head.  ``install()`` binds them
onto the reference's classes (and swaps its ``Disp`` / ``DisparityRegression``), so the growth loop
(``expand`` / ``select``), the NAS search and ``approaches/rag.py`` call the B200 path unchanged.
Everything else in the reference (2-D / 3-D convolutions, growth logic) is untouched.

``PathRouter`` is the dispatch the paper calls the Scene Router: the reference selects the grown
path with the oracle task id (``self.archis[t]``, approaches/rag.py:208,416); the router groups a
batch by a per-sample scene id and runs each group through its ``task_arch``.
"""
from __future__ import annotations

import torch

from .functional import cost_volume, disp_head
from .fused_stem import VirtualCostVolume, stem_forward
from .modules import CostVolume, Disp, DisparityRegression  # noqa: F401  (re-exported)

# Process-wide default set by install(fuse_stem=...) (every install() call sets it, so a later
# install(fuse_stem=False) switches it off again).  A network instance overrides it with the attribute
# ``rag_b200_fuse_stem`` (True / False).  When on, the patched forwards hand the Matching Net a
# VirtualCostVolume and its first layer (ConvBR_3d, made fusion-aware) runs cost volume + conv + BN + ReLU
# as one kernel; this needs ConvBR_3d.forward to be the fusion-aware one (install(fuse_stem=True) once).
_FUSE_STEM = False
_STEM_AWARE = False      # ConvBR_3d.forward has been rebound (a VirtualCostVolume may be handed out)
_ORIGINALS = {}          # (module object id, attribute path) -> original, for uninstall()


def _volume(self, x, y, maxdisp):
    fuse = getattr(self, "rag_b200_fuse_stem", None)
    if fuse is None:
        fuse = _FUSE_STEM
    if fuse and _STEM_AWARE:
        return VirtualCostVolume(x, y, maxdisp)
    return cost_volume(x, y, maxdisp)


def _head(self, cost):
    # use the module if it is already ours (keeps hooks working), else the functional form
    d = getattr(self, "disp", None)
    if isinstance(d, Disp):
        return d(cost)
    return disp_head(cost, self.maxdisp)


def network_forward(self, left, right, t, task_arch=None, path=None):
    """Replacement for Network.forward (rag_model.py:369-387)."""
    x = self.feature(left, task_arch, path)
    y = self.feature(right, task_arch, path)
    cost = _volume(self, x, y, self.maxdisp)        # rag_model.py:375-383
    cost = self.matching(cost, task_arch, path)
    return _head(self, cost)                        # rag_model.py:386


def network_search_forward(self, left, right, t, selected_ops):
    """Replacement for Network.search_forward (rag_model.py:688-706)."""
    x = self.search_feature(left, selected_ops)
    y = self.search_feature(right, selected_ops)
    cost = _volume(self, x, y, self.maxdisp)        # rag_model.py:694-702
    cost = self.search_matching(cost, selected_ops, t)
    return _head(self, cost)


def basic_network_forward(self, left, right, fea_ops, mat_ops):
    """Replacement for BasicNetwork.forward (mdenas_basicmodel.py:76-97)."""
    x = self.feature(left, fea_ops)
    y = self.feature(right, fea_ops)
    cost = cost_volume(x, y, self.maxdisp)          # mdenas_basicmodel.py:83-91 (supernet: always materialised)
    cost = self.matching(cost, mat_ops)
    return _head(self, cost)


def install(rag_model=None, mdenas_basicmodel=None, operations_3d=None, fuse_stem: bool = False, upsample: bool = False,
            matching_convs: bool = False, pointwise_convs: bool = False, resample: bool = False, resample_modules=(),
            grid_sample: bool = False, grid_sample_modules=(), matching_tf32: bool = False,
            matching_tf32_wgrad: bool = False, level12_convs: bool = False) -> dict:
    """Bind the B200 hot path onto the reference's modules (pass the imported module objects
    ``models.rag_model`` and/or ``automl.mdenas_basicmodel``).  Returns what was patched.
    New networks constructed afterwards get ``rag_b200.Disp``; existing instances keep working
    because the patched ``forward`` methods bypass ``self.disp`` when it is the reference's.

    ``fuse_stem=True`` (needs ``operations_3d`` = the imported ``automl.operations_3d``) additionally makes
    ``ConvBR_3d.forward`` fusion-aware and lets the patched forwards skip materialising the volume: the
    first Matching-Net layer (rag_model.py:341) then runs as csrc/cv_stem.cu in inference; training and
    any non-matching layer geometry fall back to the materialised volume automatically.  The same rebinding
    sends ``last_3_3d`` (a bias-free Conv3d C -> 1, 3x3x3 without BN/ReLU, rag_model.py:269) through
    csrc/last_conv.cu when no gradient is wanted (rag_b200/last_conv.py).  NOTE: only the
    growable ``Network`` starts its Matching Net with a ConvBR_3d on the raw volume in all configurations;
    the search supernet (``BasicNetwork``/``AutoMatching``) keeps the materialised volume.

    ``upsample=True`` (needs ``rag_model``) sends the ``upsample_6`` / ``upsample_12`` steps of ``matching()`` /
    ``search_matching()`` (``nn.Upsample(..., mode='trilinear', align_corners=True)``, rag_model.py:356-357,675-676) through
    csrc/trilinear.cu, forward and deterministic backward (rag_b200/upsample.py).

    ``matching_convs=True`` (needs ``operations_3d``) binds ``ConvBR_3d.forward`` to ``rag_b200.matching_conv.matching_forward``:
    the Matching Net's interior 3x3x3 ConvBR_3d layers with (C, O) in ``matching_conv.PAIRS`` (``stem3d1``, the cells'
    ``conv_3x3`` ops -- also those of the search supernet) run on csrc/conv3d_cc.cu in inference and training (folded
    BatchNorm + ReLU in eval(); batch statistics, running-estimate updates and the backward otherwise).  Every call that does
    not qualify (``matching_conv.qualifies``) goes to the ``fuse_stem`` binding unchanged, so the fused stem, ``last_3_3d``
    and the cuDNN fallback behave as without the flag.

    ``matching_tf32=True`` (needs ``matching_convs=True``, else ``ValueError``) runs those layers' convolutions on the tensor
    cores in TF32 (csrc/conv3d_cc_tf32.cu): the forward and the data gradient, while ``torch.backends.cudnn.allow_tf32`` is on
    at call time -- the precision the reference's cuDNN convolutions get by default.  BatchNorm and the weight gradient stay
    fp32.  Every install() sets it, so a later install() without it, or uninstall(), turns it off.

    ``matching_tf32_wgrad=True`` (needs ``matching_tf32=True``, else ``ValueError``) runs those layers' weight gradient in
    TF32 as well (``matching_conv.use_tf32_wgrad``: the same call-time rule), so a training step's three convolutions all
    run at cuDNN's default precision.  It changes results, so it is a flag of its own; every install() sets it too.

    ``level12_convs=True`` (needs ``matching_convs=True``, else ``ValueError``) also routes the level-12 cells' ``conv_3x3``
    op, ``ConvBR_3d(16, 16, 3, 1, 1)`` (``matching_conv.level12_qualifies``), onto the kernels, in fp32 under any TF32 flag.
    Every install() sets it, so a later install() without it, or uninstall(), turns it off.

    ``pointwise_convs=True`` (needs ``operations_3d``) binds ``ConvBR_3d.forward`` to ``rag_b200.pointwise_conv``'s
    ``pointwise_forward``: the Matching Net's pointwise ``ConvBR_3d(C, O, 1, 1, 0)`` layers (``last_12_3d``, ``last_6_3d``, the
    cells' 1x1x1 layers) that ``pointwise_conv.qualifies`` accepts run on csrc/conv3d_pw.cu in inference and training.  Every
    other call goes to the binding this call makes without the flag: ``matching_forward`` with ``matching_convs=True``,
    else ``stem_forward``.

    ``resample=True`` binds ``rag_b200.resample.FProxy()`` (``torch.nn.functional`` with ``interpolate`` replaced) as ``F`` in
    ``rag_model``, if given, and in every module of ``resample_modules`` (for the search supernet's cells:
    ``automl.build_model_2d`` and ``automl.build_model_3d``).  The cells' ``F.interpolate`` calls in ``bilinear`` (4-D) and
    ``trilinear`` (5-D) mode then run on csrc/trilinear.cu, forward and fixed-order backward, so a training step runs
    under ``torch.use_deterministic_algorithms(True)`` on the kernels; every other call is ``F.interpolate`` unchanged.  A
    module without an ``F`` attribute raises ``ValueError``, as does the flag with no module to bind.

    ``grid_sample=True`` binds ``rag_b200.grid_sample.GridSampleProxy(module.F)`` as ``F`` in every module of
    ``grid_sample_modules`` (the self-supervised variant's loss module, ``models.loss`` of ``src_self``).  Its
    ``F.grid_sample`` calls that ``grid_sample.routes`` accepts (4-D bilinear, zeros or border padding, CUDA fp32) then run on
    csrc/grid_sample.cu, forward and fixed-order backward, so the warp of the self-supervised loss runs under
    ``torch.use_deterministic_algorithms(True)``; every other call is ``F.grid_sample`` unchanged.  The proxy wraps the module's
    current ``F``, so a module bound by ``resample=True`` keeps its ``interpolate``, in either order of the two flags, and a
    module already holding a ``GridSampleProxy`` is not wrapped again.  A module without ``F`` raises ``ValueError``, as does
    the flag with no module; all modules are checked before any is bound."""
    global _FUSE_STEM, _STEM_AWARE
    if matching_tf32 and not matching_convs:
        raise ValueError("matching_tf32=True needs matching_convs=True (it selects the precision of those layers)")
    if matching_tf32_wgrad and not matching_tf32:
        raise ValueError("matching_tf32_wgrad=True needs matching_tf32=True (it extends TF32 to those layers' weight gradient)")
    if level12_convs and not matching_convs:
        raise ValueError("level12_convs=True needs matching_convs=True (it extends that binding to the 16 -> 16 layers)")
    done = {}

    def bind(owner, name, value):
        _ORIGINALS.setdefault((owner, name), getattr(owner, name))
        setattr(owner, name, value)

    if fuse_stem:
        if operations_3d is None:
            raise ValueError("fuse_stem=True needs operations_3d (the reference's automl.operations_3d module)")
        bind(operations_3d.ConvBR_3d, "forward", stem_forward)
        _STEM_AWARE = True
        done["operations_3d"] = ["ConvBR_3d.forward"]
    if matching_convs:
        if operations_3d is None:
            raise ValueError("matching_convs=True needs operations_3d (the reference's automl.operations_3d module)")
        from .matching_conv import matching_forward

        bind(operations_3d.ConvBR_3d, "forward", matching_forward)   # delegates to stem_forward: fusion-aware as well
        _STEM_AWARE = True
        done["operations_3d"] = ["ConvBR_3d.forward"]
    if pointwise_convs:
        if operations_3d is None:
            raise ValueError("pointwise_convs=True needs operations_3d (the reference's automl.operations_3d module)")
        from .pointwise_conv import pointwise_forward, pointwise_matching_forward

        bind(operations_3d.ConvBR_3d, "forward", pointwise_matching_forward if matching_convs else pointwise_forward)
        _STEM_AWARE = True
        done["operations_3d"] = ["ConvBR_3d.forward"]
    _FUSE_STEM = bool(fuse_stem)          # always (re)set: install(fuse_stem=False) after a fused install turns it off
    from .matching_conv import set_level12, set_tf32, set_tf32_wgrad

    set_tf32(matching_tf32)               # likewise
    set_tf32_wgrad(matching_tf32_wgrad)
    set_level12(level12_convs)
    if rag_model is not None:
        bind(rag_model.Network, "forward", network_forward)
        bind(rag_model.Network, "search_forward", network_search_forward)
        bind(rag_model, "Disp", Disp)
        bind(rag_model, "DisparityRegression", DisparityRegression)
        done["rag_model"] = ["Network.forward", "Network.search_forward", "Disp", "DisparityRegression"]
    if upsample:
        if rag_model is None:
            raise ValueError("upsample=True needs rag_model (the reference's models.rag_model module)")
        from .upsample import NNProxy

        bind(rag_model, "nn", NNProxy())        # `nn.Upsample(...)` inside matching() now resolves to rag_b200.upsample.Upsample
        done["rag_model"].append("nn.Upsample")
    if resample:
        targets = ([rag_model] if rag_model is not None else []) + list(resample_modules)
        if not targets:
            raise ValueError("resample=True needs rag_model or resample_modules (the reference modules whose F to bind)")
        for mod in targets:                     # all checked before any is bound
            if not hasattr(mod, "F"):
                raise ValueError(f"resample=True: module {getattr(mod, '__name__', mod)!r} has no attribute F to bind")
        from .grid_sample import GridSampleProxy
        from .resample import FProxy

        proxy = FProxy()
        for mod in targets:                     # `F.interpolate(...)` inside the cells now resolves to rag_b200.resample.interpolate
            bind(mod, "F", GridSampleProxy(proxy) if isinstance(mod.F, GridSampleProxy) else proxy)   # keeps an earlier grid_sample=True
            done.setdefault("rag_model" if mod is rag_model else getattr(mod, "__name__", repr(mod)), []).append("F.interpolate")
    if grid_sample:
        targets = list(grid_sample_modules)
        if not targets:
            raise ValueError("grid_sample=True needs grid_sample_modules (the reference modules whose F to bind, e.g. src_self's models.loss)")
        for mod in targets:                     # all checked before any is bound
            if not hasattr(mod, "F"):
                raise ValueError(f"grid_sample=True: module {getattr(mod, '__name__', mod)!r} has no attribute F to bind")
        from .grid_sample import GridSampleProxy

        for mod in targets:
            if not isinstance(mod.F, GridSampleProxy):
                bind(mod, "F", GridSampleProxy(mod.F))   # `F.grid_sample(...)` now resolves to rag_b200.grid_sample.grid_sample
            key = "rag_model" if mod is rag_model else getattr(mod, "__name__", repr(mod))
            if "F.grid_sample" not in done.setdefault(key, []):
                done[key].append("F.grid_sample")
    if mdenas_basicmodel is not None:
        bind(mdenas_basicmodel.BasicNetwork, "forward", basic_network_forward)
        bind(mdenas_basicmodel, "Disp", Disp)
        bind(mdenas_basicmodel, "DisparityRegression", DisparityRegression)
        done["mdenas_basicmodel"] = ["BasicNetwork.forward", "Disp", "DisparityRegression"]
    return done


def uninstall() -> int:
    """Undo every install(): restore the reference's own forwards / classes.  Returns how many bindings
    were restored.  (Tests use it to compare patched and unpatched networks in one process.)"""
    global _FUSE_STEM, _STEM_AWARE
    n = 0
    for (owner, name), orig in list(_ORIGINALS.items()):
        setattr(owner, name, orig)
        n += 1
    _ORIGINALS.clear()
    _FUSE_STEM = False
    _STEM_AWARE = False
    from .matching_conv import set_level12, set_tf32, set_tf32_wgrad

    set_tf32(False)
    set_tf32_wgrad(False)
    set_level12(False)
    return n


class PathRouter:
    """Scene-router dispatch over grown paths (BASELINE config 4): ``archis[u]`` is the ``task_arch``
    of scene u (what ``Network.select`` returned for task u, approaches/rag.py:101-102).  ``route``
    runs each scene's sub-batch through its path and scatters the results back in input order.
    The hot-path modules are parameter-free and shared by every path."""

    def __init__(self, model, archis):
        self.model = model
        self.archis = list(archis)

    @torch.no_grad()
    def route(self, left: torch.Tensor, right: torch.Tensor, scene_ids) -> torch.Tensor:
        scene_ids = torch.as_tensor(scene_ids)
        if scene_ids.numel() != left.shape[0]:
            raise ValueError("one scene id per stereo pair")
        out = None
        for u in sorted(set(int(s) for s in scene_ids.tolist())):
            if not 0 <= u < len(self.archis):
                raise IndexError(f"scene id {u} has no grown path (have {len(self.archis)})")
            idx = torch.nonzero(scene_ids == u).flatten().to(left.device)
            d = self.model.forward(left.index_select(0, idx).contiguous(), right.index_select(0, idx).contiguous(), u, self.archis[u])
            if out is None:
                out = torch.empty((left.shape[0],) + tuple(d.shape[1:]), dtype=d.dtype, device=d.device)
            out.index_copy_(0, idx, d)
        return out
