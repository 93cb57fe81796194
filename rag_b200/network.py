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
            matching_convs: bool = False, pointwise_convs: bool = False) -> dict:
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

    ``pointwise_convs=True`` (needs ``operations_3d``) binds ``ConvBR_3d.forward`` to ``rag_b200.pointwise_conv``'s
    ``pointwise_forward``: the Matching Net's pointwise ``ConvBR_3d(C, O, 1, 1, 0)`` layers (``last_12_3d``, ``last_6_3d``, the
    cells' 1x1x1 layers) that ``pointwise_conv.qualifies`` accepts run on csrc/conv3d_pw.cu in inference and training.  Every
    other call goes to the binding this call makes without the flag: ``matching_forward`` with ``matching_convs=True``,
    else ``stem_forward``."""
    global _FUSE_STEM, _STEM_AWARE
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
